// ingest_internal.h — the BGZF / BAI / BAM-record reader of the native ingest: the host paths of ingest.cpp, and the
// handle (file descriptor, reference dictionary, BAI chunk queries) the GPU ingest of bgzf_gpu.cu stages its blocks from.
#pragma once
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <errno.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <memory>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../include/tredsw.h"
#include "inflate_fast.h"

void tredsw_set_error(const char *fmt, ...);

namespace tredsw_ingest {

struct Bgzf {
    FILE *fh = nullptr;
    // A stream (pipe, stdin, socket) instead of a file: read strictly in order with read(), never seeked.  `sbuf` keeps
    // the compressed bytes read so far from stream offset `sbase` on, so that load() can go back to any block from there
    // on; it reads further as it needs.
    int sfd = -1;
    bool seof = false;                                // read() returned 0
    std::vector<unsigned char> sbuf;
    int64_t sbase = 0, spos = 0;
    std::vector<unsigned char> cbuf, block;
    const unsigned char *cur = nullptr;               // inflated bytes of the current block
    int64_t block_coffset = -1, next_coffset = 0;
    size_t pos = 0;
    z_stream zs;
    bool zs_init = false;
    size_t blen = 0;                                  // inflated bytes of the current block (block has slack behind)
    tredsw_inflate::FastInflater *fast = nullptr;     // own decoder (inflate_fast.h); zlib is the fallback
    long long n_fast = 0, n_zlib = 0;                 // blocks inflated by either
    // Sticky: set on I/O or format failure (a truncated or corrupt file) — NOT on a clean end of file.  Every
    // entry point that read through this handle checks it and reports TREDSW_ERR_IO instead of partial evidence.
    const char *err = nullptr;
    bool fail(const char *why) { if (!err) err = why; return false; }

    // n bytes at the current position: fread on a file; from sbuf on a stream, reading the stream further first
    size_t get(void *dst, size_t n) {
        if (sfd < 0) return fread(dst, 1, n, fh);
        while (!seof && spos + (int64_t)n > sbase + (int64_t)sbuf.size()) {
            const size_t have = sbuf.size(), want = std::max<size_t>(spos + n - sbase - have, 1 << 16);
            sbuf.resize(have + want);
            const ssize_t k = ::read(sfd, sbuf.data() + have, want);
            sbuf.resize(have + (k > 0 ? (size_t)k : 0));
            if (k == 0) seof = true;
            else if (k < 0 && errno != EINTR) { fail("read failed"); break; }
        }
        const int64_t avail = std::max<int64_t>(0, sbase + (int64_t)sbuf.size() - spos);
        const size_t take = std::min<size_t>(n, (size_t)avail);
        if (take) memcpy(dst, sbuf.data() + (spos - sbase), take);
        spos += (int64_t)take;
        return take;
    }
    bool at_eof() { return sfd < 0 ? feof(fh) != 0 : seof && spos >= sbase + (int64_t)sbuf.size(); }

    bool load(int64_t coffset) {
        blen = 0; pos = 0; block_coffset = coffset; next_coffset = coffset;
        if (sfd >= 0) { if (coffset < sbase) return fail("the stream has moved past this block"); spos = coffset; }
        else if (fseeko(fh, coffset, SEEK_SET) != 0) return fail("seek failed");
        unsigned char head[18];
        const size_t nhead = get(head, 18);
        if (nhead == 0 && at_eof()) return false;                          // clean end of file
        if (nhead != 18) return fail("truncated BGZF block header");
        if (head[0] != 31 || head[1] != 139 || !(head[3] & 4)) return fail("not a BGZF block");
        const int xlen = head[10] | (head[11] << 8);
        std::vector<unsigned char> extra(xlen);
        memcpy(extra.data(), head + 12, std::min(6, xlen));
        if (xlen > 6 && get(extra.data() + 6, xlen - 6) != (size_t)(xlen - 6)) return fail("truncated BGZF block header");
        int bsize = -1;
        for (int off = 0; off + 4 <= xlen;) {
            const int slen = extra[off + 2] | (extra[off + 3] << 8);
            if (extra[off] == 66 && extra[off + 1] == 67 && off + 6 <= xlen) bsize = extra[off + 4] | (extra[off + 5] << 8);
            off += 4 + slen;
        }
        if (bsize < 0) return fail("BGZF block without a BC field");
        const int clen = bsize - xlen - 19;
        if (clen < 0) return fail("bad BGZF block size");
        cbuf.resize(clen > 0 ? clen : 0);
        if (clen > 0 && get(cbuf.data(), clen) != (size_t)clen) return fail("truncated BGZF block");
        unsigned char tail[8];
        if (get(tail, 8) != 8) return fail("truncated BGZF block");
        const uint32_t crc = tail[0] | (tail[1] << 8) | (tail[2] << 16) | ((uint32_t)tail[3] << 24);
        const uint32_t isize = tail[4] | (tail[5] << 8) | (tail[6] << 16) | ((uint32_t)tail[7] << 24);
        if (isize > 65536) return fail("BGZF block larger than 64 KiB");   // (the format's limit; also bounds the resize)
        if (block.size() < (size_t)isize + tredsw_inflate::FastInflater::SLACK) block.resize((size_t)isize + tredsw_inflate::FastInflater::SLACK);
        blen = isize;
        cur = block.data();
        if (isize > 0) {
            static const bool zlib_only = getenv("TREDSW_ZLIB_INFLATE") != nullptr;
            bool done = false;
            if (!zlib_only && clen > 0) {
                if (!fast) fast = new tredsw_inflate::FastInflater();
                // the block's CRC-32 guards the result: anything else than a verified block goes to zlib
                done = fast->inflate(cbuf.data(), (size_t)clen, block.data(), isize) &&
                       (uint32_t)crc32(crc32(0L, Z_NULL, 0), block.data(), isize) == crc;
                if (done) ++n_fast;
            }
            if (!done) {
                if (!zs_init) { memset(&zs, 0, sizeof(zs)); if (inflateInit2(&zs, -15) != Z_OK) { blen = 0; return fail("zlib init failed"); } zs_init = true; }
                else inflateReset(&zs);
                zs.next_in = cbuf.data(); zs.avail_in = (uInt)clen;
                zs.next_out = block.data(); zs.avail_out = isize;
                const int rc = inflate(&zs, Z_FINISH);
                if (rc != Z_STREAM_END || zs.total_out != isize ||
                    (uint32_t)crc32(crc32(0L, Z_NULL, 0), block.data(), isize) != crc) { blen = 0; return fail("corrupt BGZF block (inflate / length / CRC-32)"); }
                ++n_zlib;
            }
        }
        next_coffset = coffset + bsize + 1;
        return true;
    }
    void seek(uint64_t voffset) {
        const int64_t coffset = (int64_t)(voffset >> 16);
        if (coffset != block_coffset) load(coffset);
        pos = (size_t)(voffset & 0xffff);
    }
    uint64_t tell() const {
        if (pos >= blen && block_coffset >= 0) return (uint64_t)next_coffset << 16;
        return ((uint64_t)block_coffset << 16) | pos;
    }
    size_t read(void *dst, size_t n) {
        unsigned char *out = (unsigned char *)dst;
        size_t got = 0;
        while (n > 0) {
            size_t avail = blen > pos ? blen - pos : 0;
            if (avail == 0) {
                const int64_t prev = block_coffset;
                if (!load(next_coffset)) break;
                if (blen == 0) { if (next_coffset == block_coffset || block_coffset == prev) break; continue; }
                avail = blen;
            }
            const size_t take = std::min(avail, n);
            memcpy(out + got, cur + pos, take);
            pos += take; got += take; n -= take;
        }
        return got;
    }
    ~Bgzf() { if (zs_init) inflateEnd(&zs); if (fh) fclose(fh); if (sfd >= 0) close(sfd); delete fast; }
};

struct RefIndex {
    std::unordered_map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins;
    std::vector<uint64_t> linear;
};

struct Record {
    int32_t tid, pos, next_tid, next_pos, tlen, l_seq;
    uint16_t flag;
    int32_t ref_len;          // reference span of the CIGAR
    int32_t qstart, qend;     // query_alignment_start / _end (soft clips)
    bool has_cigar;
    std::string name;
    const unsigned char *seq; // packed 4-bit, valid until the next record is read
};

}  // namespace tredsw_ingest

struct tredsw_bam {
    typedef tredsw_ingest::Bgzf Bgzf;
    typedef tredsw_ingest::RefIndex RefIndex;
    typedef tredsw_ingest::Record Record;
    Bgzf bgzf;
    std::vector<std::string> names;
    std::vector<int64_t> lengths;
    std::unordered_map<std::string, int32_t> tid_of;
    // the parsed .bai (tens of MB for a whole-genome BAM) is immutable and shared by the clones of a handle
    std::shared_ptr<const std::vector<RefIndex>> index_ptr;
    std::string path;
    std::string text;                // the header text (SAM header lines)
    bool has_index = false;
    bool consumed = false;           // a stream handle whose scan has read the stream (it can be read only once)
    uint64_t first_record = 0;       // virtual offset of the first alignment record
    bool is_stream() const { return bgzf.sfd >= 0; }
    std::vector<unsigned char> rec;

    bool read_record(Record &r) {
        int32_t bs;
        const size_t nbs = bgzf.read(&bs, 4);
        if (nbs == 0) return false;                                          // end of file (or bgzf.err)
        if (nbs != 4) return bgzf.fail("truncated BAM record");
        if (bs < 32 || bs > (64 << 20)) return bgzf.fail("bad BAM record size");
        rec.resize(bs);
        if (bgzf.read(rec.data(), bs) != (size_t)bs) return bgzf.fail("truncated BAM record");
        const unsigned char *d = rec.data();
        auto i32 = [&](int o) { int32_t v; memcpy(&v, d + o, 4); return v; };
        auto u16 = [&](int o) { uint16_t v; memcpy(&v, d + o, 2); return v; };
        r.tid = i32(0); r.pos = i32(4);
        const int l_name = d[8];
        const int n_cigar = u16(12);
        r.flag = u16(14); r.l_seq = i32(16); r.next_tid = i32(20); r.next_pos = i32(24); r.tlen = i32(28);
        // a record whose variable-length fields do not fit its block_size is corrupt: stop reading
        if (r.l_seq < 0 || 32LL + l_name + 4LL * n_cigar + ((int64_t)r.l_seq + 1) / 2 + r.l_seq > (int64_t)bs) return bgzf.fail("corrupt BAM record");
        int off = 32;
        r.name.assign((const char *)d + off, l_name > 0 ? l_name - 1 : 0);
        off += l_name;
        r.ref_len = 0; r.has_cigar = n_cigar > 0;
        int qs = 0, qe = r.l_seq;
        bool lead = true;
        for (int k = 0; k < n_cigar; ++k) {
            uint32_t c; memcpy(&c, d + off + 4 * k, 4);
            const int op = c & 15, len = (int)(c >> 4);
            if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) r.ref_len += len;   // M D N = X
            if (lead) { if (op == 4) qs += len; else if (op != 5) lead = false; }
        }
        for (int k = n_cigar - 1; k >= 0; --k) {
            uint32_t c; memcpy(&c, d + off + 4 * k, 4);
            const int op = c & 15, len = (int)(c >> 4);
            if (op == 4) qe -= len; else if (op != 5) break;
        }
        r.qstart = qs; r.qend = qe;
        off += 4 * n_cigar;
        r.seq = d + off;
        return true;
    }

    // merged chunk list of an indexed region query (same rule as bamio.BAIIndex.chunks)
    std::vector<std::pair<uint64_t, uint64_t>> chunks(int tid, int64_t beg, int64_t end) const {
        std::vector<std::pair<uint64_t, uint64_t>> out;
        if (!index_ptr || tid < 0 || tid >= (int)index_ptr->size()) return out;
        const RefIndex &ri = (*index_ptr)[tid];
        uint64_t min_off = 0;
        if (!ri.linear.empty()) { const size_t k = (size_t)(beg >> 14); min_off = k < ri.linear.size() ? ri.linear[k] : ri.linear.back(); }
        const int64_t e1 = end - 1;
        auto add_bin = [&](uint32_t b) {
            if (b == 37450) return;
            auto it = ri.bins.find(b);
            if (it == ri.bins.end()) return;
            for (auto &c : it->second) if (c.second > min_off) out.push_back(c);
        };
        add_bin(0);
        const int shifts[5] = {26, 23, 20, 17, 14}, offs[5] = {1, 9, 73, 585, 4681};
        for (int l = 0; l < 5; ++l)
            for (int64_t b = offs[l] + (beg >> shifts[l]); b <= offs[l] + (e1 >> shifts[l]); ++b) add_bin((uint32_t)b);
        std::sort(out.begin(), out.end());
        std::vector<std::pair<uint64_t, uint64_t>> merged;
        for (auto &c : out) {
            if (!merged.empty() && c.first <= merged.back().second) merged.back().second = std::max(merged.back().second, c.second);
            else merged.push_back(c);
        }
        return merged;
    }

    // records overlapping [start, end) on tid, in file order (bamio.AlignmentFile._iter_indexed)
    template <class F>
    void fetch(int tid, int64_t start, int64_t end, F &&fn) {
        if (start < 0) start = 0;
        Record r;
        for (auto &c : chunks(tid, start, end)) {
            bgzf.seek(c.first);
            while (bgzf.tell() < c.second) {
                if (!read_record(r)) break;
                if (r.tid != tid) { if (r.tid >= 0 && r.tid < tid) continue; return; }
                if (r.pos >= end) return;
                int64_t rend = (int64_t)r.pos + r.ref_len;
                if ((r.flag & 4) || !r.has_cigar || rend <= r.pos) rend = (int64_t)r.pos + 1;
                if (r.pos < end && rend > start) fn(r);
            }
        }
    }
};

