// Streaming host BAM reader: BGZF blocks inflated on a thread pool, records decoded contig by contig (or region by
// region through the .bai linear index) straight into the flat packed read arrays (struct nsnp_reads).
//
// This is the "host decodes the BAM into flat packed arrays" step of the north star; it replaces the BAM reading that
// `samtools mpileup` does for the reference (make_predict_data.sh:151).  Nothing is held but one batch of inflated
// blocks (<= 32 MB) and the arrays of the contig / region being decoded.  Formats: SAM/BAM specification sections
// 4.1 (BGZF), 4.2 (BAM records, CG:B,I long CIGARs) and 5.2 (BAI).  Host code only (zlib); no GPU work here.
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <atomic>
#include <chrono>
#include <future>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

namespace {

inline int32_t rd_i32(const uint8_t* p) { int32_t v; memcpy(&v, p, 4); return v; }
inline uint32_t rd_u32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
inline uint16_t rd_u16(const uint8_t* p) { uint16_t v; memcpy(&v, p, 2); return v; }
inline uint64_t rd_u64(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }

struct Block { const uint8_t* cdata; uint32_t clen, isize; };

// one BGZF member at p: fills b, returns the member's total size, 0 at a clean end, -1 when malformed
int64_t bgzf_member(const uint8_t* p, const uint8_t* lim, Block* b) {
    if (p == lim) return 0;
    if (lim - p < 18 || p[0] != 31 || p[1] != 139 || p[2] != 8 || !(p[3] & 4)) return -1;
    const uint32_t xlen = rd_u16(p + 10);
    if (p + 12 + xlen > lim) return -1;
    int64_t bsize = -1;
    for (uint32_t o = 0; o + 4 <= xlen;) {
        const uint8_t* x = p + 12 + o;
        const uint32_t slen = rd_u16(x + 2);
        if (x[0] == 66 && x[1] == 67 && slen == 2) bsize = rd_u16(x + 4);
        o += 4 + slen;
    }
    if (bsize < 0) return -1;
    const int64_t total = bsize + 1;
    if (total < 12 + (int64_t)xlen + 8 || p + total > lim) return -1;
    b->cdata = p + 12 + xlen;
    b->clen = (uint32_t)(total - 12 - xlen - 8);
    b->isize = rd_u32(p + total - 4);
    return total;
}

struct Batch { std::vector<uint8_t> data; bool ok = true; bool eof = false; };

// 4-bit BAM base codes "=ACMGRSVTWYHKDBN": one input byte (two bases) -> low nibble = two 2-bit codes, bits 4/5 = N flags.
// '=' and the IUPAC ambiguity codes count like N: `samtools mpileup` prints them verbatim and the tensor maker only
// counts ACGTacgt (tensor_maker.cpp:104-107).
struct NibbleLut {
    uint8_t v[256];
    NibbleLut() {
        static const int8_t c2[16] = {-1, 0, 1, -1, 2, -1, -1, -1, 3, -1, -1, -1, -1, -1, -1, -1};
        for (int b = 0; b < 256; ++b) {
            const int hi = b >> 4, lo = b & 15;        // the first base is the high nibble
            v[b] = (uint8_t)((c2[hi] < 0 ? 0 : c2[hi]) | ((c2[lo] < 0 ? 0 : c2[lo]) << 2) | ((c2[hi] < 0) << 4) | ((c2[lo] < 0) << 5));
        }
    }
};
const NibbleLut g_lut;

struct BaiRef { uint64_t first = 0; bool has = false; std::vector<uint64_t> ioff; };

}  // namespace

struct nsnp_bam_reader {
    int fd = -1;
    const uint8_t* file = nullptr; size_t file_len = 0;
    int n_threads = 1;
    // stream state
    size_t next_block = 0;                  // file offset of the next BGZF member to inflate
    int batch_blocks = 8;                   // read-ahead ramps up from 8 blocks (0.5 MB) to 512 (32 MB); reset by seek()
    std::vector<uint8_t> buf; size_t cur = 0;
    std::future<Batch> pending; bool pending_valid = false, at_eof = false;
    // header
    std::vector<std::string> ref_names; std::vector<int64_t> ref_lens;
    // index
    bool has_bai = false; std::vector<BaiRef> bai;
    // decoded arrays of the current contig / region
    std::vector<int32_t> pos; std::vector<uint16_t> flag; std::vector<uint8_t> mapq;
    std::vector<int64_t> cigar_off, seq_off; std::vector<uint32_t> cigar; std::vector<uint8_t> seq2, nmask;
    int64_t n_bases = 0; bool any_n = false;
    bool keep_aux = false;                  // HaplotypeModel s4: also keep base qualities, HP tag and a query-name hash
    std::vector<uint8_t> qual, hp; std::vector<uint64_t> qhash;
    int64_t inflated_bytes = 0;
    double t_wait = 0, t_buf = 0, t_fill = 0;     // seconds: waiting for inflate, buffer upkeep, record fill (NSNP_TRACE)
    static double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

    Batch inflate_batch(size_t from, int max_blocks, size_t* next_out) {
        Batch out;
        std::vector<Block> blocks; std::vector<size_t> off;
        size_t o = from, total = 0;
        const uint8_t* lim = file + file_len;
        while ((int)blocks.size() < max_blocks && total < (32u << 20)) {
            Block b;
            const int64_t used = bgzf_member(file + o, lim, &b);
            if (used == 0) { out.eof = true; break; }
            if (used < 0) { out.ok = false; break; }
            off.push_back(total); blocks.push_back(b); total += b.isize; o += (size_t)used;
        }
        *next_out = o;
        out.data.resize(total);
        std::atomic<size_t> ticket{0}; std::atomic<bool> good{true};
        auto work = [&]() {
            z_stream zs; memset(&zs, 0, sizeof zs);
            if (inflateInit2(&zs, -15) != Z_OK) { good = false; return; }
            for (;;) {
                const size_t i = ticket.fetch_add(1);
                if (i >= blocks.size()) break;
                if (blocks[i].isize == 0) continue;
                inflateReset(&zs);
                zs.next_in = const_cast<Bytef*>(blocks[i].cdata); zs.avail_in = blocks[i].clen;
                zs.next_out = out.data.data() + off[i]; zs.avail_out = blocks[i].isize;
                const int rc = inflate(&zs, Z_FINISH);
                if (rc != Z_STREAM_END || zs.avail_out != 0) { good = false; break; }
            }
            inflateEnd(&zs);
        };
        const int nt = (int)std::min<size_t>((size_t)n_threads, std::max<size_t>(1, blocks.size() / 8));
        std::vector<std::thread> th;
        for (int t = 1; t < nt; ++t) th.emplace_back(work);
        work();
        for (auto& t : th) t.join();
        if (!good) out.ok = false;
        return out;
    }

    void launch_next() {
        if (at_eof) return;
        const size_t from = next_block;
        // the batch boundary is found synchronously (cheap header walk) so that next_block is known at once
        size_t o = from, total = 0; int nb = 0;
        const uint8_t* lim = file + file_len;
        const int max_blocks = batch_blocks;
        batch_blocks = std::min(512, batch_blocks * 2);
        while (nb < max_blocks && total < (32u << 20)) {
            Block b; const int64_t used = bgzf_member(file + o, lim, &b);
            if (used <= 0) break;
            total += b.isize; o += (size_t)used; ++nb;
        }
        next_block = o;
        pending = std::async(std::launch::async, [this, from, max_blocks]() { size_t dummy; return inflate_batch(from, max_blocks, &dummy); });
        pending_valid = true;
    }

    // makes at least n bytes available at buf[cur..]; false at end of stream / error (err set on corruption)
    bool need(size_t n, bool* err) {
        while (buf.size() - cur < n) {
            if (!pending_valid) { if (at_eof) return false; launch_next(); }
            double t0 = now();
            Batch b = pending.get(); pending_valid = false;
            t_wait += now() - t0;
            if (!b.ok) { *err = true; return false; }
            flush_pending();                                     // queued records point into buf
            t0 = now();
            if (cur > 0) { buf.erase(buf.begin(), buf.begin() + (ptrdiff_t)cur); cur = 0; }
            buf.insert(buf.end(), b.data.begin(), b.data.end());
            t_buf += now() - t0;
            inflated_bytes += (int64_t)b.data.size();
            if (b.eof || next_block >= file_len) at_eof = true;
            else launch_next();                                  // the next batch inflates while this one is parsed
        }
        return true;
    }

    void seek(uint64_t voff) {
        if (pending_valid) { pending.get(); pending_valid = false; }
        flush_pending();
        buf.clear(); cur = 0; at_eof = false; batch_blocks = 8;
        next_block = (size_t)(voff >> 16);
        bool err = false;
        const size_t u = (size_t)(voff & 0xffff);
        need(u, &err);
        cur = std::min(u, buf.size());
    }

    void clear_arrays() {
        pos.clear(); flag.clear(); mapq.clear(); cigar_off.assign(1, 0); seq_off.clear(); cigar.clear();
        seq2.clear(); nmask.clear(); qual.clear(); hp.clear(); qhash.clear(); n_bases = 0; any_n = false; pend.clear(); pend_cig = 0; pend_bases = 0; merge_needed = false;
    }

    // ---- decode: records are indexed sequentially (cheap: header fields only), then filled by all threads ----
    struct RecRef { const uint8_t* p; const uint8_t* cg; const uint8_t* seq; uint32_t nc, l_seq; int64_t cig_o, base_o; const uint8_t* aux; const uint8_t* end; };
    std::vector<RecRef> pend;
    int64_t pend_cig = 0, pend_bases = 0;
    bool merge_needed = false;

    // value of the HP:i tag (whatshap haplotag: 1 or 2), 0 when absent; walks the aux fields per the SAM spec
    static uint8_t aux_hp(const uint8_t* t, const uint8_t* end) {
        while (t + 3 <= end) {
            const char a = (char)t[0], b = (char)t[1], ty = (char)t[2];
            t += 3; size_t sz = 0;
            if (ty == 'A' || ty == 'c' || ty == 'C') sz = 1;
            else if (ty == 's' || ty == 'S') sz = 2;
            else if (ty == 'i' || ty == 'I' || ty == 'f') sz = 4;
            else if (ty == 'Z' || ty == 'H') { const uint8_t* e = t; while (e < end && *e) ++e; sz = (size_t)(e - t) + 1; }
            else if (ty == 'B') {
                if (t + 5 > end) return 0;
                const char sub = (char)t[0]; const uint32_t cnt = rd_u32(t + 1);
                sz = 5 + (size_t)((sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4) * cnt;
            } else return 0;
            if (t + sz > end) return 0;
            if (a == 'H' && b == 'P') {
                int64_t v = 0;
                switch (ty) { case 'c': v = (int8_t)t[0]; break; case 'C': v = t[0]; break; case 's': v = (int16_t)rd_u16(t); break;
                              case 'S': v = rd_u16(t); break; case 'i': v = rd_i32(t); break; case 'I': v = rd_u32(t); break; default: v = 0; }
                return (v >= 0 && v <= 255) ? (uint8_t)v : 0;
            }
            t += sz;
        }
        return 0;
    }

    // queues the record at p (block_size bytes after the 4-byte length)
    void queue(const uint8_t* p, int64_t bs) {
        const uint32_t l_name = p[12], n_cig_rec = rd_u16(p + 16), l_seq = rd_u32(p + 20);
        const uint8_t* q = p + 36 + l_name;
        const uint8_t* cg = q; uint32_t nc = n_cig_rec;
        q += 4ull * n_cig_rec;
        const uint8_t* seq = q; q += (l_seq + 1) / 2 + l_seq;
        const uint8_t* end = p + 4 + bs;
        if (nc == 2) {                      // CG:B,I long CIGAR (placeholder <l_seq>S<ref_len>N in the record)
            const uint32_t c0 = rd_u32(cg), c1 = rd_u32(cg + 4);
            if ((c0 & 15) == 4 && (c0 >> 4) == l_seq && (c1 & 15) == 3) {
                const uint8_t* t = q;
                while (t + 3 <= end) {
                    const char a = (char)t[0], b = (char)t[1], ty = (char)t[2];
                    t += 3; size_t sz = 0;
                    if (ty == 'A' || ty == 'c' || ty == 'C') sz = 1;
                    else if (ty == 's' || ty == 'S') sz = 2;
                    else if (ty == 'i' || ty == 'I' || ty == 'f') sz = 4;
                    else if (ty == 'Z' || ty == 'H') { const uint8_t* e = t; while (e < end && *e) ++e; sz = (size_t)(e - t) + 1; }
                    else if (ty == 'B') {
                        if (t + 5 > end) break;
                        const char sub = (char)t[0]; const uint32_t cnt = rd_u32(t + 1);
                        const size_t es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
                        if (a == 'C' && b == 'G' && sub == 'I' && t + 5 + 4ull * cnt <= end) { cg = t + 5; nc = cnt; break; }
                        sz = 5 + es * cnt;
                    } else break;
                    t += sz;
                }
            }
        }
        const int64_t padded = ((int64_t)l_seq + 15) / 16 * 16;     // every read starts on a 16-base boundary of seq2 / nmask
        pend.push_back(RecRef{p, cg, seq, nc, l_seq, (int64_t)cigar.size() + pend_cig, n_bases + pend_bases, q, end});
        pend_cig += nc; pend_bases += padded;
    }

    // fills the arrays from the queued records (must run before the bytes they point into are released)
    void flush_pending() {
        if (pend.empty()) return;
        const double t_begin = now();
        const size_t n0 = pos.size(), nr = pend.size();
        pos.resize(n0 + nr); flag.resize(n0 + nr); mapq.resize(n0 + nr); seq_off.resize(n0 + nr); cigar_off.resize(n0 + nr + 1);
        cigar.resize(cigar.size() + (size_t)pend_cig);
        seq2.resize(seq2.size() + (size_t)pend_bases / 4, 0); nmask.resize(nmask.size() + (size_t)pend_bases / 8, 0);
        if (keep_aux) { qual.resize(qual.size() + (size_t)pend_bases, 0); hp.resize(n0 + nr, 0); qhash.resize(n0 + nr, 0); }
        std::atomic<size_t> ticket{0};
        std::atomic<bool> saw_n{false}, need_merge{false};
        auto work = [&]() {
            bool my_n = false, my_merge = false;
            for (;;) {
                const size_t i0 = ticket.fetch_add(16);
                if (i0 >= nr) break;
                for (size_t i = i0; i < std::min(nr, i0 + 16); ++i) {
                    const RecRef& r = pend[i];
                    pos[n0 + i] = rd_i32(r.p + 8); flag[n0 + i] = rd_u16(r.p + 18); mapq[n0 + i] = r.p[13];
                    seq_off[n0 + i] = r.base_o; cigar_off[n0 + i + 1] = r.cig_o + r.nc;
                    uint32_t* c = cigar.data() + r.cig_o;
                    memcpy(c, r.cg, 4ull * r.nc);
                    for (uint32_t k = 1; k < r.nc; ++k) my_merge |= ((c[k] ^ c[k - 1]) & 15u) == 0;
                    uint8_t* s2 = seq2.data() + r.base_o / 4; uint8_t* nm = nmask.data() + r.base_o / 8;
                    const uint32_t nb = (r.l_seq + 1) / 2;
                    uint32_t nacc = 0, j = 0;
                    for (; j + 4 <= nb; j += 4) {                        // 8 bases: two seq2 bytes, one nmask byte
                        const uint32_t v0 = g_lut.v[r.seq[j]], v1 = g_lut.v[r.seq[j + 1]], v2 = g_lut.v[r.seq[j + 2]], v3 = g_lut.v[r.seq[j + 3]];
                        s2[j >> 1] = (uint8_t)((v0 & 15) | ((v1 & 15) << 4)); s2[(j >> 1) + 1] = (uint8_t)((v2 & 15) | ((v3 & 15) << 4));
                        const uint32_t nf = (v0 >> 4) | ((v1 >> 4) << 2) | ((v2 >> 4) << 4) | ((v3 >> 4) << 6);
                        nm[j >> 2] = (uint8_t)nf; nacc |= nf;
                    }
                    for (; j < nb; ++j) {
                        const uint32_t v = g_lut.v[r.seq[j]];
                        s2[j >> 1] |= (uint8_t)((v & 15) << (4 * (j & 1)));
                        nm[j >> 2] |= (uint8_t)((v >> 4) << (2 * (j & 3)));
                        nacc |= v >> 4;
                    }
                    if (r.l_seq & 1) {                                  // odd length: the last low nibble is padding, not a base
                        const uint32_t k = r.l_seq;                     // index of the phantom base
                        s2[k >> 2] &= (uint8_t)~(3u << (2 * (k & 3)));
                        const bool was = (nm[k >> 3] >> (k & 7)) & 1u;
                        nm[k >> 3] &= (uint8_t)~(1u << (k & 7));
                        if (was) {                                      // recompute: the phantom may have been the only N
                            nacc = 0;
                            for (uint32_t q = 0; q < (r.l_seq + 7) / 8; ++q) nacc |= nm[q];
                        }
                    }
                    if (nacc) my_n = true;
                    if (keep_aux) {
                        memcpy(qual.data() + r.base_o, r.seq + nb, r.l_seq);
                        uint64_t hsh = 1469598103934665603ull;                     // FNV-1a of the query name (without the NUL)
                        for (const uint8_t* c = r.p + 36; *c; ++c) hsh = (hsh ^ *c) * 1099511628211ull;
                        qhash[n0 + i] = hsh;
                        hp[n0 + i] = aux_hp(r.aux, r.end);
                    }
                }
            }
            if (my_n) saw_n = true;
            if (my_merge) need_merge = true;
        };
        const int nt = (int)std::min<size_t>((size_t)n_threads, std::max<size_t>(1, nr / 32));
        std::vector<std::thread> th;
        for (int t = 1; t < nt; ++t) th.emplace_back(work);
        work();
        for (auto& t : th) t.join();
        if (saw_n) any_n = true;
        if (need_merge) merge_needed = true;
        n_bases += pend_bases;
        pend.clear(); pend_cig = 0; pend_bases = 0;
        t_fill += now() - t_begin;
    }

    // adjacent ops of one type merged ("1D2D" -> "3D": htslib reports such runs as one indel); rare, so a sequential pass
    void merge_runs() {
        if (!merge_needed) return;
        size_t w = 0;
        for (size_t r = 0; r + 1 < cigar_off.size(); ++r) {
            const size_t b = (size_t)cigar_off[r], e = (size_t)cigar_off[r + 1], w0 = w;
            for (size_t k = b; k < e; ++k) {
                if (w > w0 && ((cigar[w - 1] ^ cigar[k]) & 15u) == 0) cigar[w - 1] += cigar[k] & ~15u;
                else cigar[w++] = cigar[k];
            }
            cigar_off[r] = (int64_t)w0;
        }
        cigar_off[cigar_off.size() - 1] = (int64_t)w;
        cigar.resize(w);
        merge_needed = false;
    }
};

extern "C" {

nsnp_bam_reader_t* nsnp_bam_open(const char* path, int n_threads)
{
    if (!path) { nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_open: null path"); return nullptr; }
    nsnp_bam_reader* r = new nsnp_bam_reader();
    r->n_threads = n_threads > 0 ? n_threads : (int)std::max(1u, std::thread::hardware_concurrency());
    r->fd = open(path, O_RDONLY);
    struct stat st;
    if (r->fd < 0 || fstat(r->fd, &st) != 0) { nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_open: cannot open %s", path); delete r; return nullptr; }
    r->file_len = (size_t)st.st_size;
    void* m = r->file_len ? mmap(nullptr, r->file_len, PROT_READ, MAP_PRIVATE, r->fd, 0) : nullptr;
    if (r->file_len && m == MAP_FAILED) { nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_open: mmap failed for %s", path); close(r->fd); delete r; return nullptr; }
    r->file = (const uint8_t*)m;
    if (m) madvise(m, r->file_len, MADV_SEQUENTIAL);
    bool err = false;
    auto fail = [&](const char* what) { nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_open: %s: %s", path, what); nsnp_bam_close(r); return (nsnp_bam_reader_t*)nullptr; };
    if (!r->need(12, &err) || memcmp(r->buf.data() + r->cur, "BAM\1", 4) != 0) return fail("not a BAM stream");
    const int64_t l_text = rd_i32(r->buf.data() + r->cur + 4);
    if (l_text < 0 || !r->need(12 + (size_t)l_text, &err)) return fail("truncated header");
    r->cur += 8 + (size_t)l_text;
    const int32_t n_ref = rd_i32(r->buf.data() + r->cur); r->cur += 4;
    for (int32_t i = 0; i < n_ref; ++i) {
        if (!r->need(4, &err)) return fail("truncated reference list");
        const int32_t l_name = rd_i32(r->buf.data() + r->cur);
        if (l_name < 1 || !r->need(8 + (size_t)l_name, &err)) return fail("truncated reference list");
        r->ref_names.emplace_back((const char*)r->buf.data() + r->cur + 4, (size_t)l_name - 1);
        r->ref_lens.push_back(rd_i32(r->buf.data() + r->cur + 4 + l_name));
        r->cur += 8 + (size_t)l_name;
    }
    // optional index: <path>.bai or <stem>.bai
    std::string p1 = std::string(path) + ".bai", p2 = path;
    if (p2.size() > 4 && p2.substr(p2.size() - 4) == ".bam") p2 = p2.substr(0, p2.size() - 4) + ".bai";
    for (const std::string& bp : {p1, p2}) {
        FILE* f = fopen(bp.c_str(), "rb");
        if (!f) continue;
        std::vector<uint8_t> d; uint8_t tmp[65536]; size_t k;
        while ((k = fread(tmp, 1, sizeof tmp, f)) > 0) d.insert(d.end(), tmp, tmp + k);
        fclose(f);
        size_t o = 8; bool ok = d.size() >= 8 && memcmp(d.data(), "BAI\1", 4) == 0 && rd_i32(d.data() + 4) == n_ref;
        std::vector<BaiRef> refs((size_t)std::max(0, n_ref));
        for (int32_t i = 0; ok && i < n_ref; ++i) {
            if (o + 4 > d.size()) { ok = false; break; }
            const int32_t n_bin = rd_i32(d.data() + o); o += 4;
            uint64_t first = ~0ull;
            for (int32_t b = 0; ok && b < n_bin; ++b) {
                if (o + 8 > d.size()) { ok = false; break; }
                const uint32_t bin = rd_u32(d.data() + o); const int32_t n_chunk = rd_i32(d.data() + o + 4); o += 8;
                if (o + 16ull * (size_t)n_chunk > d.size()) { ok = false; break; }
                if (bin != 37450) for (int32_t c = 0; c < n_chunk; ++c) first = std::min(first, rd_u64(d.data() + o + 16ull * c));
                o += 16ull * (size_t)n_chunk;
            }
            if (!ok || o + 4 > d.size()) { ok = false; break; }
            const int32_t n_intv = rd_i32(d.data() + o); o += 4;
            if (o + 8ull * (size_t)n_intv > d.size()) { ok = false; break; }
            refs[i].ioff.resize((size_t)n_intv);
            for (int32_t k2 = 0; k2 < n_intv; ++k2) refs[i].ioff[k2] = rd_u64(d.data() + o + 8ull * k2);
            o += 8ull * (size_t)n_intv;
            refs[i].has = first != ~0ull; refs[i].first = first;
        }
        if (ok) { r->bai.swap(refs); r->has_bai = true; break; }
    }
    return r;
}

void nsnp_bam_close(nsnp_bam_reader_t* r)
{
    if (!r) return;
    if (getenv("NSNP_TRACE")) fprintf(stderr, "bam reader: inflated %.0f MB; waited for inflate %.3f s, buffer upkeep %.3f s, record fill %.3f s\n", r->inflated_bytes / 1e6, r->t_wait, r->t_buf, r->t_fill);
    if (r->pending_valid) { r->pending.get(); r->pending_valid = false; }
    if (r->file) munmap((void*)r->file, r->file_len);
    if (r->fd >= 0) close(r->fd);
    delete r;
}

int32_t nsnp_bam_n_ref(const nsnp_bam_reader_t* r) { return r ? (int32_t)r->ref_names.size() : -1; }
const char* nsnp_bam_ref_name(const nsnp_bam_reader_t* r, int32_t i) { return (r && i >= 0 && i < (int32_t)r->ref_names.size()) ? r->ref_names[i].c_str() : nullptr; }
int64_t nsnp_bam_ref_len(const nsnp_bam_reader_t* r, int32_t i) { return (r && i >= 0 && i < (int32_t)r->ref_lens.size()) ? r->ref_lens[i] : -1; }
int nsnp_bam_has_index(const nsnp_bam_reader_t* r) { return r && r->has_bai; }
int64_t nsnp_bam_inflated_bytes(const nsnp_bam_reader_t* r) { return r ? r->inflated_bytes : -1; }

// shared record loop: decodes records of reference `ref` with pos < end whose reference span reaches beyond beg.
// ref < 0: take the reference of the first wanted record.  Stops (without consuming) at the first record of another
// reference or with pos >= end.  Returns the reference decoded, -1 at end of file, -2 on corruption.
// append: keep the records already decoded (nsnp_bam_fetch_ranges)
static int32_t decode_run(nsnp_bam_reader* r, int32_t ref, const int8_t* want, int64_t beg, int64_t end, bool append = false)
{
    if (!append) r->clear_arrays();
    bool err = false;
    int32_t cur_ref = ref;
    for (;;) {
        if (!r->need(4, &err)) break;
        const int64_t bs = rd_i32(r->buf.data() + r->cur);
        if (bs < 32) { err = true; break; }
        if (!r->need(4 + (size_t)bs, &err)) { err = true; break; }
        const uint8_t* p = r->buf.data() + r->cur;
        const int32_t rid = rd_i32(p + 4), pos = rd_i32(p + 8);
        if (cur_ref < 0) {
            if (rid < 0) { r->cur += 4 + (size_t)bs; continue; }                     // unplaced reads (sorted last)
            if (want && !want[rid]) {
                // skip this reference: through the index when there is one, record by record otherwise
                int32_t nxt = -1;
                for (int32_t k = rid + 1; k < (int32_t)r->ref_names.size(); ++k)
                    if (want[k] && (!r->has_bai || r->bai[k].has)) { nxt = k; break; }
                if (r->has_bai) {
                    if (nxt < 0) return -1;
                    r->seek(r->bai[nxt].first);
                    continue;
                }
                r->cur += 4 + (size_t)bs;
                continue;
            }
            cur_ref = rid;
        }
        if (rid != cur_ref || pos >= end) break;
        const uint32_t l_name = p[12], n_cig = rd_u16(p + 16), l_seq = rd_u32(p + 20);
        if (36ull + l_name + 4ull * n_cig + (l_seq + 1) / 2 + l_seq > (uint64_t)bs + 4) { err = true; break; }
        if (beg > 0) {
            // skip reads that end before the window (the in-record CIGAR has the right reference length even when it is
            // the <l_seq>S<ref_len>N placeholder of a CG-tag long CIGAR)
            int64_t reflen = 0;
            const uint8_t* cg = p + 36 + l_name;
            for (uint32_t k = 0; k < n_cig; ++k) {
                const uint32_t c = rd_u32(cg + 4ull * k), op = c & 15u;
                if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) reflen += c >> 4;
            }
            if (pos + std::max<int64_t>(reflen, 1) <= beg) { r->cur += 4 + (size_t)bs; continue; }
        }
        r->queue(p, bs);
        r->cur += 4 + (size_t)bs;
    }
    r->flush_pending();
    r->merge_runs();
    if (err) { nsnp::set_error(NSNP_E_INVALID, "malformed BAM record stream"); return -2; }
    if (cur_ref < 0 || (r->pos.empty() && ref < 0)) return -1;
    return cur_ref;
}

int32_t nsnp_bam_next_contig(nsnp_bam_reader_t* r, const int8_t* want, int64_t* n_reads, int64_t* n_cigar, int64_t* n_bases_padded)
{
    if (!r) return -2;
    const int32_t rid = decode_run(r, -1, want, 0, INT64_MAX);
    if (n_reads) *n_reads = (int64_t)r->pos.size();
    if (n_cigar) *n_cigar = (int64_t)r->cigar.size();
    if (n_bases_padded) *n_bases_padded = r->n_bases;
    return rid;
}

int32_t nsnp_bam_fetch(nsnp_bam_reader_t* r, int32_t ref_id, int64_t beg, int64_t end, int64_t* n_reads, int64_t* n_cigar, int64_t* n_bases_padded)
{
    if (!r || ref_id < 0 || ref_id >= (int32_t)r->ref_names.size()) { nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_fetch: bad reference id"); return -2; }
    if (!r->has_bai) { nsnp::set_error(NSNP_E_UNSUPPORTED, "nsnp_bam_fetch needs a .bai index next to the BAM"); return -2; }
    r->clear_arrays();
    int32_t rid = ref_id;
    if (r->bai[ref_id].has) {
        // linear index: smallest virtual offset of any alignment overlapping the 16 kb window of `beg`
        const auto& io = r->bai[ref_id].ioff;
        uint64_t v = 0;
        const size_t w = (size_t)(std::max<int64_t>(beg, 0) >> 14);
        if (w < io.size()) v = io[w];
        if (v == 0) { for (size_t k = std::min(w, io.size()); k-- > 0;) if (io[k]) { v = io[k]; break; } }
        if (v == 0) v = r->bai[ref_id].first;
        r->seek(v);
        // records of earlier references cannot appear after this offset; skip reads that end before the window
        rid = decode_run(r, ref_id, nullptr, beg, end);
        if (rid == -2) return -2;
    }
    if (n_reads) *n_reads = (int64_t)r->pos.size();
    if (n_cigar) *n_cigar = (int64_t)r->cigar.size();
    if (n_bases_padded) *n_bases_padded = r->n_bases;
    return ref_id;
}

int32_t nsnp_bam_fetch_ranges(nsnp_bam_reader_t* r, int32_t ref_id, const int64_t* ranges, int64_t n, int64_t* n_reads,
                              int64_t* n_cigar, int64_t* n_bases_padded)
{
    if (!r || ref_id < 0 || ref_id >= (int32_t)r->ref_names.size()) { nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_fetch_ranges: bad reference id"); return -2; }
    if (!r->has_bai) { nsnp::set_error(NSNP_E_UNSUPPORTED, "nsnp_bam_fetch_ranges needs a .bai index next to the BAM"); return -2; }
    if (n < 0 || (n > 0 && !ranges)) { nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_fetch_ranges: bad range list"); return -2; }
    for (int64_t k = 0; k < n; ++k)
        if (ranges[2 * k] < 0 || ranges[2 * k + 1] <= ranges[2 * k] || (k && ranges[2 * k] < ranges[2 * k - 1])) {
            nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_fetch_ranges: range %lld is empty, unsorted or overlapping", (long long)k);
            return -2;
        }
    r->clear_arrays();
    if (r->bai[ref_id].has) {
        const auto& io = r->bai[ref_id].ioff;
        for (int64_t k = 0; k < n; ++k) {
            const int64_t beg = ranges[2 * k], end = ranges[2 * k + 1];
            uint64_t v = 0;
            const size_t w = (size_t)(beg >> 14);
            if (w < io.size()) v = io[w];
            if (v == 0) { for (size_t j = std::min(w, io.size()); j-- > 0;) if (io[j]) { v = io[j]; break; } }
            if (v == 0) v = r->bai[ref_id].first;
            // Records are consumed in file order, so none is decoded twice.  Blocks before next_block are inflated (or being
            // inflated) already: walk on from the current record, skipping those that end before the range.  Seek only past them.
            if (k == 0 || (size_t)(v >> 16) >= r->next_block) r->seek(v);
            if (decode_run(r, ref_id, nullptr, beg, end, true) == -2) return -2;
        }
    }
    if (n_reads) *n_reads = (int64_t)r->pos.size();
    if (n_cigar) *n_cigar = (int64_t)r->cigar.size();
    if (n_bases_padded) *n_bases_padded = r->n_bases;
    return ref_id;
}

int nsnp_bam_take(nsnp_bam_reader_t* r, int32_t* pos, uint16_t* flag, uint8_t* mapq, int64_t* cigar_off, uint32_t* cigar,
                  int64_t* seq_off, uint8_t* seq2, uint8_t* nmask, int32_t* any_n)
{
    if (!r || !pos || !flag || !mapq || !cigar_off || !cigar || !seq_off || !seq2) return nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_take: null argument");
    const size_t n = r->pos.size();
    if (n) {
        memcpy(pos, r->pos.data(), n * 4); memcpy(flag, r->flag.data(), n * 2); memcpy(mapq, r->mapq.data(), n);
        memcpy(seq_off, r->seq_off.data(), n * 8);
    }
    memcpy(cigar_off, r->cigar_off.data(), (n + 1) * 8);
    if (!r->cigar.empty()) memcpy(cigar, r->cigar.data(), r->cigar.size() * 4);
    if (!r->seq2.empty()) memcpy(seq2, r->seq2.data(), r->seq2.size());
    if (nmask && !r->nmask.empty()) memcpy(nmask, r->nmask.data(), r->nmask.size());
    if (any_n) *any_n = r->any_n ? 1 : 0;
    return NSNP_OK;
}

int nsnp_bam_keep_aux(nsnp_bam_reader_t* r, int keep)
{
    if (!r) return nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_keep_aux: null reader");
    r->keep_aux = keep != 0;
    return NSNP_OK;
}

int nsnp_bam_take_aux(nsnp_bam_reader_t* r, uint8_t* qual, uint8_t* hp, uint64_t* qname_hash)
{
    if (!r || !qual || !hp || !qname_hash) return nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_take_aux: null argument");
    if (!r->keep_aux || r->hp.size() != r->pos.size()) return nsnp::set_error(NSNP_E_INVALID, "nsnp_bam_take_aux: call nsnp_bam_keep_aux(reader, 1) before decoding");
    if (!r->qual.empty()) memcpy(qual, r->qual.data(), r->qual.size());
    if (!r->hp.empty()) { memcpy(hp, r->hp.data(), r->hp.size()); memcpy(qname_hash, r->qhash.data(), r->qhash.size() * 8); }
    return NSNP_OK;
}

}  // extern "C"
