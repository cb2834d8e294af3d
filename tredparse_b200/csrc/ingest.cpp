// ingest.cpp — native BAM ingest for the genotyping path (host code, zlib only).
//
// Replaces, for one locus, the three pysam passes of the reference:
//   BamParser.parse selection .......... tredparse/bam_parser.py:194-243  (window fetch, READ window, alts)
//   PEextractor ......................... tredparse/bam_parser.py:316-369  (+-10 kb pair distances)
//   BamDepth.region_depth ............... tredparse/bam_parser.py:404-411  (pileup depth of the +-1 kb window)
// with ONE indexed pass over the BGZF blocks of the +-10 kb window, writing the reads as base codes
// (A,C,G,T,N -> 0..4, src/ssw_wrap.py:229-244), the pair distances and the depth straight into caller-owned
// (pinned) buffers — the layout tredsw_genotype_batch consumes.  Record order, pairing rule and depth
// definition are those of the Python host path (tredparse_b200/bam_parser.py, bamio.py), which the tests use
// as the oracle of this file.
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <fcntl.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <memory>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>
#include <thread>

#include "ingest_internal.h"


using namespace tredsw_ingest;

extern "C" {

// the handle with its header read (reference dictionary, first record), no index yet.  stream: read the input strictly
// in order ("-" is stdin)
static tredsw_bam *open_header(const char *bam_path, bool stream = false) {
    if (!bam_path) { tredsw_set_error("null path"); return nullptr; }
    tredsw_bam *b = new tredsw_bam();
    if (!stream) b->bgzf.fh = fopen(bam_path, "rb");
    else b->bgzf.sfd = strcmp(bam_path, "-") == 0 ? dup(STDIN_FILENO) : open(bam_path, O_RDONLY | O_CLOEXEC);
    if (!b->bgzf.fh && b->bgzf.sfd < 0) { tredsw_set_error("cannot open %s", bam_path); delete b; return nullptr; }
    char magic[4];
    int32_t l_text = 0, n_ref = 0;
    if (b->bgzf.read(magic, 4) != 4 || memcmp(magic, "BAM\1", 4) != 0 || b->bgzf.read(&l_text, 4) != 4 || l_text < 0) {
        tredsw_set_error("%s is not a BAM file", bam_path); delete b; return nullptr;
    }
    b->text.resize(l_text);
    if (l_text && b->bgzf.read(&b->text[0], l_text) != (size_t)l_text) { tredsw_set_error("truncated BAM header"); delete b; return nullptr; }
    b->text.resize(strnlen(b->text.c_str(), b->text.size()));          // (the text may end in NULs)
    if (b->bgzf.read(&n_ref, 4) != 4 || n_ref < 0) { tredsw_set_error("truncated BAM header"); delete b; return nullptr; }
    for (int i = 0; i < n_ref; ++i) {
        int32_t l_name = 0, l_ref = 0;
        if (b->bgzf.read(&l_name, 4) != 4 || l_name <= 0 || l_name > 4096) { tredsw_set_error("bad reference name"); delete b; return nullptr; }
        std::vector<char> nm(l_name);
        if (b->bgzf.read(nm.data(), l_name) != (size_t)l_name || b->bgzf.read(&l_ref, 4) != 4) { tredsw_set_error("truncated BAM header"); delete b; return nullptr; }
        b->names.emplace_back(nm.data());
        b->lengths.push_back(l_ref);
        b->tid_of[b->names.back()] = i;
    }
    b->first_record = b->bgzf.tell();
    b->path = bam_path;
    if (stream) {
        if (b->path == "-") b->path = "(stdin)";
        // the header's blocks are not needed again: keep the stream from the block of the first record on
        Bgzf &z = b->bgzf;
        const int64_t drop = std::min<int64_t>((int64_t)(b->first_record >> 16) - z.sbase, (int64_t)z.sbuf.size());
        if (drop > 0) { z.sbuf.erase(z.sbuf.begin(), z.sbuf.begin() + drop); z.sbase += drop; }
    }
    return b;
}

tredsw_bam *tredsw_bam_open_unindexed(const char *bam_path) { return open_header(bam_path); }

// A BAM read strictly in order (a pipe, stdin as "-", a socket; a regular file works the same way): no seek, no size.
// The handle keeps the compressed bytes it has read from the block of the first record on; the scan starts with them.
tredsw_bam *tredsw_bam_open_stream(const char *path) { return open_header(path, true); }

int64_t tredsw_bam_header_text(tredsw_bam *b, char *buf, int64_t cap) {
    if (!b) { tredsw_set_error("null handle"); return TREDSW_ERR_ARG; }
    if (buf && cap > 0) {
        const size_t n = std::min<size_t>(b->text.size(), (size_t)cap - 1);
        memcpy(buf, b->text.data(), n);
        buf[n] = 0;
    }
    return (int64_t)b->text.size();
}

tredsw_bam *tredsw_bam_open(const char *bam_path, const char *bai_path) {
    tredsw_bam *b = open_header(bam_path);
    if (!b) return nullptr;
    // index: <bam>.bai, then <bam without extension>.bai (bamio.AlignmentFile)
    std::string cands[2];
    if (bai_path) cands[0] = bai_path;
    else {
        cands[0] = std::string(bam_path) + ".bai";
        std::string p(bam_path);
        const size_t dot = p.rfind('.');
        cands[1] = (dot == std::string::npos ? p : p.substr(0, dot)) + ".bai";
    }
    for (const std::string &cand : cands) {
        if (cand.empty()) continue;
        FILE *fi = fopen(cand.c_str(), "rb");
        if (!fi) continue;
        fseeko(fi, 0, SEEK_END);
        const int64_t sz = ftello(fi);
        fseeko(fi, 0, SEEK_SET);
        std::vector<unsigned char> data(sz > 0 ? sz : 0);
        const bool ok = sz >= 8 && fread(data.data(), 1, sz, fi) == (size_t)sz && memcmp(data.data(), "BAI\1", 4) == 0;
        fclose(fi);
        if (!ok) continue;
        size_t off = 4;
        auto need = [&](size_t n) { return off + n <= data.size(); };
        int32_t nr = 0;
        memcpy(&nr, data.data() + off, 4); off += 4;
        bool good = true;
        auto index = std::make_shared<std::vector<RefIndex>>(nr > 0 ? nr : 0);
        for (int i = 0; i < nr && good; ++i) {
            int32_t n_bin = 0;
            if (!need(4)) { good = false; break; }
            memcpy(&n_bin, data.data() + off, 4); off += 4;
            for (int k = 0; k < n_bin; ++k) {
                uint32_t bin; int32_t n_chunk;
                if (!need(8)) { good = false; break; }
                memcpy(&bin, data.data() + off, 4); memcpy(&n_chunk, data.data() + off + 4, 4); off += 8;
                if (n_chunk < 0 || !need((size_t)16 * n_chunk)) { good = false; break; }
                auto &v = (*index)[i].bins[bin];
                for (int c = 0; c < n_chunk; ++c) {
                    uint64_t s, e;
                    memcpy(&s, data.data() + off, 8); memcpy(&e, data.data() + off + 8, 8); off += 16;
                    v.emplace_back(s, e);
                }
            }
            int32_t n_intv = 0;
            if (!good || !need(4)) { good = false; break; }
            memcpy(&n_intv, data.data() + off, 4); off += 4;
            if (n_intv < 0 || !need((size_t)8 * n_intv)) { good = false; break; }
            (*index)[i].linear.resize(n_intv);
            if (n_intv) memcpy((*index)[i].linear.data(), data.data() + off, (size_t)8 * n_intv);
            off += (size_t)8 * n_intv;
        }
        if (good) { b->index_ptr = index; b->has_index = true; break; }
    }
    if (!b->has_index) { tredsw_set_error("no usable .bai index next to %s", bam_path); delete b; return nullptr; }
    return b;
}

// A second handle on the same BAM for another host thread: its own file descriptor and inflate state, the
// header tables copied, the parsed index shared.  Handles are not thread-safe; clones are independent.
tredsw_bam *tredsw_bam_clone(tredsw_bam *src) {
    if (!src) { tredsw_set_error("null handle"); return nullptr; }
    if (src->is_stream()) { tredsw_set_error("%s is a stream: it can be read only once, by one handle", src->path.c_str()); return nullptr; }
    tredsw_bam *b = new tredsw_bam();
    b->bgzf.fh = fopen(src->path.c_str(), "rb");
    if (!b->bgzf.fh) { tredsw_set_error("cannot open %s", src->path.c_str()); delete b; return nullptr; }
    b->names = src->names; b->lengths = src->lengths; b->tid_of = src->tid_of;
    b->index_ptr = src->index_ptr; b->has_index = src->has_index;
    b->first_record = src->first_record; b->path = src->path; b->text = src->text;
    return b;
}

void tredsw_bam_close(tredsw_bam *b) { delete b; }

// BGZF blocks inflated by this handle so far: by the library's own decoder / by zlib (the fallback).
// A signature of the reference dictionary (names and lengths in order): handles with equal signatures number their
// contigs alike, so per-locus queries built for one sample of a cohort can be reused for the next.
uint64_t tredsw_bam_header_signature(tredsw_bam *b) {
    if (!b) return 0;
    uint64_t h = 1469598103934665603ull;
    auto mix = [&](const void *p, size_t n) { const unsigned char *c = (const unsigned char *)p; for (size_t i = 0; i < n; ++i) { h ^= c[i]; h *= 1099511628211ull; } };
    for (size_t i = 0; i < b->names.size(); ++i) { mix(b->names[i].c_str(), b->names[i].size() + 1); mix(&b->lengths[i], sizeof(b->lengths[i])); }
    return h ? h : 1;
}

void tredsw_bam_inflate_stats(tredsw_bam *b, int64_t *own, int64_t *zlib_blocks) {
    if (own) *own = b ? b->bgzf.n_fast : 0;
    if (zlib_blocks) *zlib_blocks = b ? b->bgzf.n_zlib : 0;
}

// The raw-DEFLATE decoder on its own (test hook): 0 when `in` inflates to exactly out_len bytes.
int tredsw_inflate_raw(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_len) {
    if (!in || !out || in_len < 0 || out_len < 0) return TREDSW_ERR_ARG;
    std::vector<uint8_t> buf((size_t)out_len + tredsw_inflate::FastInflater::SLACK);
    tredsw_inflate::FastInflater dec;
    if (!dec.inflate(in, (size_t)in_len, buf.data(), (size_t)out_len)) return TREDSW_ERR_UNSUPPORTED;
    memcpy(out, buf.data(), (size_t)out_len);
    return TREDSW_OK;
}

int32_t tredsw_bam_nref(tredsw_bam *b) { return b ? (int32_t)b->names.size() : 0; }

int64_t tredsw_bam_ref(tredsw_bam *b, int32_t tid, char *name, int64_t cap) {
    if (!b || tid < 0 || tid >= (int32_t)b->names.size()) return -1;
    const std::string &n = b->names[tid];
    if (name && cap > 0) {
        const size_t k = std::min<size_t>(n.size(), (size_t)cap - 1);
        memcpy(name, n.data(), k);
        name[k] = 0;
    }
    return b->lengths[tid];
}

int32_t tredsw_bam_tid(tredsw_bam *b, const char *name) {
    if (!b || !name) return -1;
    auto it = b->tid_of.find(name);
    return it == b->tid_of.end() ? -1 : it->second;
}

// BamDepth.region_depth (bam_parser.py:404-411): sum of pileup column depths / (end - start + 1).  pysam's
// default pileup walks every column of every qualifying read overlapping the window, so the column sum is the
// total reference span of the overlapping reads that are not UNMAP / SECONDARY / QCFAIL / DUP
// (same restatement as bamio.region_depth).
int tredsw_bam_region_depth(tredsw_bam *b, int32_t tid, int64_t start, int64_t end, double *depth) {
    if (!b || !depth) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (b->is_stream()) { tredsw_set_error("%s is a stream: region queries need an indexed file", b->path.c_str()); return TREDSW_ERR_UNSUPPORTED; }
    if (!b->has_index) { tredsw_set_error("%s has no index", b->path.c_str()); return TREDSW_ERR_UNSUPPORTED; }
    if (tid < 0 || tid >= (int)b->names.size()) { tredsw_set_error("contig id %d out of range", tid); return TREDSW_ERR_ARG; }
    if (end < start) { tredsw_set_error("empty region"); return TREDSW_ERR_ARG; }
    int64_t total = 0;
    b->bgzf.err = nullptr;
    try {
        b->fetch(tid, start, end, [&](const Record &r) {
            if ((r.flag & (4 | 256 | 512 | 1024)) || !r.has_cigar) return;
            total += r.ref_len;
        });
    } catch (const std::exception &e) { tredsw_set_error("tredsw_bam_region_depth: %s", e.what()); return TREDSW_ERR_IO; }
    if (b->bgzf.err) { tredsw_set_error("%s: %s", b->path.c_str(), b->bgzf.err); return TREDSW_ERR_IO; }
    *depth = (double)total * 1.0 / (double)(end - start + 1);
    return TREDSW_OK;
}

// BamReadLen.readlen (bam_parser.py:372-391): the longest query among the first `first_n` + 1 records of the
// file (the reference breaks after len(rls) > firstN); min_out may be NULL.  On a stream these records are read ahead
// and stay buffered for the scan.
int tredsw_bam_read_length(tredsw_bam *b, int32_t first_n, int32_t *max_out, int32_t *min_out) {
    if (!b || !max_out || first_n < 0) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (b->consumed) { tredsw_set_error("%s: stream already consumed", b->path.c_str()); return TREDSW_ERR_ARG; }
    int32_t n = 0, mx = -1, mn = 0x7fffffff;
    b->bgzf.err = nullptr;
    try {
        b->bgzf.seek(b->first_record);
        Record r;
        while (n <= first_n && b->read_record(r)) {
            mx = std::max(mx, r.l_seq); mn = std::min(mn, r.l_seq);
            ++n;
        }
    } catch (const std::exception &e) { tredsw_set_error("tredsw_bam_read_length: %s", e.what()); return TREDSW_ERR_IO; }
    if (b->bgzf.err) { tredsw_set_error("%s: %s", b->path.c_str(), b->bgzf.err); return TREDSW_ERR_IO; }
    if (n == 0) { tredsw_set_error("no records"); return TREDSW_ERR_ARG; }
    *max_out = mx;
    if (min_out) *min_out = mn;
    return TREDSW_OK;
}

static int extract_locus_impl(tredsw_bam *b, const tredsw_locus_query *q, int8_t *rbuf, int64_t rbuf_cap,
                              int64_t *roff, int32_t reads_cap, int32_t *global_lens, int32_t global_cap,
                              int32_t *target_lens, int32_t target_cap, char *names, int64_t names_cap,
                              tredsw_locus_summary *out);

int tredsw_bam_extract_locus(tredsw_bam *b, const tredsw_locus_query *q, int8_t *rbuf, int64_t rbuf_cap,
                             int64_t *roff, int32_t reads_cap, int32_t *global_lens, int32_t global_cap,
                             int32_t *target_lens, int32_t target_cap, char *names, int64_t names_cap,
                             tredsw_locus_summary *out) {
    if (!b || !q || !out || !roff || reads_cap < 0) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (b->is_stream()) { tredsw_set_error("%s is a stream: region queries need an indexed file", b->path.c_str()); return TREDSW_ERR_UNSUPPORTED; }
    if (!b->has_index) { tredsw_set_error("%s has no index", b->path.c_str()); return TREDSW_ERR_UNSUPPORTED; }
    b->bgzf.err = nullptr;
    int rc;
    try {
        rc = extract_locus_impl(b, q, rbuf, rbuf_cap, roff, reads_cap, global_lens, global_cap, target_lens, target_cap,
                                names, names_cap, out);
    } catch (const std::exception &e) { tredsw_set_error("tredsw_bam_extract_locus: %s", e.what()); return TREDSW_ERR_IO; }
    // a truncated or corrupt file must not come back as "fewer reads": no partial evidence
    if (rc == TREDSW_OK && b->bgzf.err) { tredsw_set_error("%s: %s", b->path.c_str(), b->bgzf.err); memset(out, 0, sizeof(*out)); return TREDSW_ERR_IO; }
    return rc;
}

static int extract_locus_impl(tredsw_bam *b, const tredsw_locus_query *q, int8_t *rbuf, int64_t rbuf_cap,
                              int64_t *roff, int32_t reads_cap, int32_t *global_lens, int32_t global_cap,
                              int32_t *target_lens, int32_t target_cap, char *names, int64_t names_cap,
                              tredsw_locus_summary *out) {
    if (q->tid < 0 || q->tid >= (int)b->names.size()) { tredsw_set_error("contig id %d out of range", q->tid); return TREDSW_ERR_ARG; }
    static const int8_t NIB[16] = {4, 0, 1, 4, 2, 4, 4, 4, 3, 4, 4, 4, 4, 4, 4, 4};   // "=ACMGRSVTWYHKDBN"
    memset(out, 0, sizeof(*out));
    const int64_t start = q->repeat_start, end = q->repeat_end;
    const int64_t WIN_S = std::max<int64_t>(0, start - q->pad), WIN_E = end + q->pad;               // parse window
    const int64_t READ_S = std::max<int64_t>(0, start - q->readlen), READ_E = end + q->readlen;
    const int64_t PE_S = std::max<int64_t>(start - q->pe_window, 0), PE_E = end + q->pe_window;     // pair window
    const int64_t tstart = start - q->flankmatch, tend = end + q->flankmatch;
    int64_t nbases = 0, name_bytes = 0, depth_sum = 0;
    int32_t nreads = 0;
    roff[0] = 0;
    auto emit_read = [&](const Record &r) {
        if (nreads < reads_cap && nbases + r.l_seq <= rbuf_cap && rbuf) {
            int8_t *dst = rbuf + nbases;
            for (int i = 0; i < r.l_seq; ++i) dst[i] = NIB[(r.seq[i >> 1] >> ((i & 1) ? 0 : 4)) & 15];
            roff[nreads + 1] = nbases + r.l_seq;
        } else out->overflow = 1;
        if (names) {
            if (name_bytes + (int64_t)r.name.size() + 1 <= names_cap) { memcpy(names + name_bytes, r.name.c_str(), r.name.size() + 1); }
            else out->overflow = 1;
        }
        name_bytes += (int64_t)r.name.size() + 1;
        nbases += r.l_seq;
        ++nreads;
    };
    // pairs of the +-pe_window region, keyed by name in order of first appearance (PEextractor)
    struct Mate { int32_t pos, ref_end, qstart, qend, l_seq; bool reverse; };
    std::unordered_map<std::string, int> slot;
    std::vector<std::pair<Mate, Mate>> pairs;
    std::vector<int> npair;
    const int64_t lo = std::min(WIN_S, PE_S), hi = std::max(WIN_E, PE_E);
    b->fetch(q->tid, lo, hi, [&](const Record &r) {
        int64_t rend = (int64_t)r.pos + r.ref_len;
        const bool unmapped = (r.flag & 4) != 0;
        if (unmapped || !r.has_cigar || rend <= r.pos) rend = (int64_t)r.pos + 1;
        // (1) reads handed to Smith-Waterman: overlap the +-pad window; mapped ones must start in the READ window
        if (r.pos < WIN_E && rend > WIN_S) {
            if (unmapped) { ++out->n_unmapped; emit_read(r); }
            else if (r.pos >= READ_S && r.pos <= READ_E) emit_read(r);
            // (3) pileup depth of the +-pad window: reference span of every counted read that overlaps it
            if (!(r.flag & (4 | 256 | 512 | 1024)) && r.has_cigar) depth_sum += r.ref_len;
        }
        // (2) properly paired, mapped, non-duplicate records of the pair window
        if (r.pos < PE_E && rend > PE_S && (r.flag & 1) && !unmapped && !(r.flag & 1024)) {
            auto it = slot.find(r.name);
            Mate m{r.pos, (int32_t)((r.flag & 4) || !r.has_cigar ? -1 : r.pos + r.ref_len), r.qstart, r.qend, r.l_seq, (r.flag & 16) != 0};
            if (it == slot.end()) { slot.emplace(r.name, (int)pairs.size()); pairs.emplace_back(m, Mate{}); npair.push_back(1); }
            else if (npair[it->second] == 1) { pairs[it->second].second = m; npair[it->second] = 2; }
            else ++npair[it->second];
        }
    });
    // alt regions: reads whose MATE lies in the parse window of this locus (bam_parser.py:215-243)
    for (int a = 0; a < q->n_alts && q->alts; ++a) {
        const int32_t atid = q->alts[3 * a], as = q->alts[3 * a + 1], ae = q->alts[3 * a + 2];
        if (atid < 0 || atid >= (int)b->names.size()) continue;
        b->fetch(atid, as, ae, [&](const Record &r) {
            if (r.next_tid != q->tid) return;
            if (r.next_pos < WIN_S || r.next_pos > WIN_E) return;
            emit_read(r);
        });
    }
    int32_t ng = 0, nt = 0;
    for (size_t i = 0; i < pairs.size(); ++i) {
        if (npair[i] < 2) continue;
        const Mate &x = pairs[i].first, &y = pairs[i].second;
        if (!(!x.reverse && y.reverse)) continue;
        int64_t s = x.pos, e = y.ref_end;
        if (x.qstart > 0) s -= x.qstart;
        if (y.qend < y.l_seq) e += y.l_seq - y.qend;
        const int64_t tlen = e - s;
        if (tlen >= q->span) continue;
        if (x.pos < tstart && y.ref_end > tend) { if (nt < target_cap && target_lens) target_lens[nt] = (int32_t)tlen; else out->overflow = 1; ++nt; }
        else { if (ng < global_cap && global_lens) global_lens[ng] = (int32_t)tlen; else out->overflow = 1; ++ng; }
    }
    out->nreads = nreads; out->nbases = nbases; out->name_bytes = name_bytes;
    out->n_global = ng; out->n_target = nt;
    out->depth = (double)depth_sum * 1.0 / (double)(WIN_E - WIN_S + 1);
    return TREDSW_OK;
}


}  // extern "C"

#if defined(__x86_64__)
#include <immintrin.h>
// 64 codes -> 32 bytes per iteration: maddubs(lo, hi) x (1, 16) = lo | hi << 4 in every 16-bit lane, then pack
__attribute__((target("avx2"))) static int64_t pack4_avx2(const int8_t *codes, int64_t nbytes_out, uint8_t *out) {
    const __m256i mask = _mm256_set1_epi8(0x0F), mul = _mm256_set1_epi16(0x1001);
    int64_t b = 0;
    for (; b + 32 <= nbytes_out; b += 32) {
        __m256i x0 = _mm256_and_si256(_mm256_loadu_si256(reinterpret_cast<const __m256i *>(codes + 2 * b)), mask);
        __m256i x1 = _mm256_and_si256(_mm256_loadu_si256(reinterpret_cast<const __m256i *>(codes + 2 * b + 32)), mask);
        x0 = _mm256_maddubs_epi16(x0, mul);
        x1 = _mm256_maddubs_epi16(x1, mul);
        const __m256i p = _mm256_permute4x64_epi64(_mm256_packus_epi16(x0, x1), 0xD8);
        _mm256_storeu_si256(reinterpret_cast<__m256i *>(out + b), p);
    }
    return b;
}
static bool have_avx2() { static const bool v = __builtin_cpu_supports("avx2"); return v; }
#else
static int64_t pack4_avx2(const int8_t *, int64_t, uint8_t *) { return 0; }
static bool have_avx2() { return false; }
#endif

extern "C" {

// ---- host-side transfer formats (tredsw_cohort.input_flags) ------------------------------------------------------
// Two base codes per byte / int16 pair lengths: what a cohort pipeline does to every batch between ingest and the
// host-to-device copy.  Plain loops (the compiler vectorises them), split over `threads` std::threads.
int tredsw_pack_reads4(const int8_t *codes, int64_t n, uint8_t *out, int threads) {
    if ((!codes && n > 0) || !out || n < 0) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    const int64_t nbytes = (n + 1) / 2;
    // 8 codes (one 64-bit word) -> 4 bytes with shifts and masks only, so that the loop vectorises
    auto work = [&](int64_t b0, int64_t b1) {                    // output bytes [b0, b1), b0 a multiple of 4
        int64_t b = b0;
        if (have_avx2() && 2 * b1 <= n) b += pack4_avx2(codes + 2 * b0, b1 - b0, out + b0);
        for (; b + 4 <= b1 && 2 * b + 8 <= n; b += 4) {
            uint64_t x;
            memcpy(&x, codes + 2 * b, 8);
            x &= 0x0F0F0F0F0F0F0F0FULL;
            x = (x | (x >> 4)) & 0x00FF00FF00FF00FFULL;         // bytes 0, 2, 4, 6: lo | hi << 4
            x = (x | (x >> 8)) & 0x0000FFFF0000FFFFULL;
            x = (x | (x >> 16));
            const uint32_t y = (uint32_t)x;
            memcpy(out + b, &y, 4);
        }
        for (; b < b1; ++b) {
            const int64_t i = 2 * b;
            const unsigned lo = (unsigned)codes[i] & 15u, hi = (i + 1 < n) ? ((unsigned)codes[i + 1] & 15u) : 0u;
            out[b] = (uint8_t)(lo | (hi << 4));
        }
    };
    if (threads <= 1 || nbytes < (1 << 20)) { work(0, nbytes); return TREDSW_OK; }
    try {
        std::vector<std::thread> pool;
        const int64_t per = ((nbytes + threads - 1) / threads + 3) & ~(int64_t)3;
        for (int t = 0; t < threads; ++t) {
            const int64_t b0 = (int64_t)t * per, b1 = std::min(nbytes, b0 + per);
            if (b0 < b1) pool.emplace_back(work, b0, b1);
        }
        for (auto &th : pool) th.join();
    } catch (const std::exception &e) { tredsw_set_error("tredsw_pack_reads4: %s", e.what()); return TREDSW_ERR_ARG; }
    return TREDSW_OK;
}

int tredsw_narrow_i16(const int32_t *in, int64_t n, int16_t *out, int threads) {
    if ((!in && n > 0) || !out || n < 0) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    // branch-free body (vectorises); the range check is an OR over the block
    auto work = [&](int64_t a, int64_t b, int *bad) {
        int32_t acc = 0;
        for (int64_t i = a; i < b; ++i) {
            const int32_t v = in[i];
            acc |= (v + 32768) & ~0xFFFF;
            out[i] = (int16_t)v;
        }
        *bad = acc != 0;
    };
    int nt = (threads <= 1 || n < (1 << 20)) ? 1 : threads;
    std::vector<int> bad((size_t)nt, 0);
    if (nt == 1) work(0, n, &bad[0]);
    else {
        try {
            std::vector<std::thread> pool;
            const int64_t per = (n + nt - 1) / nt;
            for (int t = 0; t < nt; ++t) {
                const int64_t a = (int64_t)t * per, b = std::min(n, a + per);
                if (a < b) pool.emplace_back(work, a, b, &bad[(size_t)t]);
            }
            for (auto &th : pool) th.join();
        } catch (const std::exception &e) { tredsw_set_error("tredsw_narrow_i16: %s", e.what()); return TREDSW_ERR_ARG; }
    }
    for (int b : bad) if (b) { tredsw_set_error("a pair length does not fit int16"); return TREDSW_ERR_ARG; }
    return TREDSW_OK;
}

}  // extern "C"
