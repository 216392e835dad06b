// bam.cpp — BAM input (SAMv1 §4): the decoded image of a BAM file, its SAM text, and the BGZF writer of the synthetic data.
//
// A BAM file is BGZF (gzip members of at most 64 KiB, each with a "BC" extra field holding its compressed size) around the
// stream  "BAM\1" l_text text n_ref {l_name name l_ref}*  {block_size record}*.  The image built here - the inflated stream,
// the offset of every record, the refID -> contig table, the header's line count - is the one decoded form both parsers use:
//   the host packer (sam_pack.cpp) parses the records' SAM lines rendered by bam_to_sam;
//   the device decoder (tok_kernels.cu) uploads the image and runs bam_rec.h one record per thread.
// Which SAM line a record stands for: SAMv1 §4.2's columns, with QUAL written as "*" (polish never reads it) and of the
// optional fields only those polish reads (NM of an integer type as NM:i, ZP:Z, alignment.rs:67-75); a CG:B:I array replaces
// the long-CIGAR placeholder kSmN.
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <thread>

#include "pp_internal.h"
#include "bam_rec.h"

namespace pp {

namespace {

constexpr uint32_t BGZF_MAX = 65536;
constexpr size_t PAD = 64;                  // zero bytes behind the stream (the byte reader loads whole 8-byte words)

inline uint32_t rd16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }
inline uint32_t rd32(const uint8_t* p) { return rd16(p) | (rd16(p + 2) << 16); }

// The BGZF block header at p (n bytes available): its total size (BSIZE + 1) and where its extra field ends, or 0.
uint32_t bgzf_block(const uint8_t* p, size_t n, uint32_t* xlen_out) {
    if (n < 18 || p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return 0;
    const uint32_t xlen = rd16(p + 10);
    if (n < 12 + (size_t)xlen) return 0;
    for (uint32_t q = 12; q + 4 <= 12 + xlen;) {
        const uint32_t slen = rd16(p + q + 2);
        if (p[q] == 'B' && p[q + 1] == 'C' && slen == 2 && q + 6 <= 12 + xlen) {
            const uint32_t bsize = rd16(p + q + 4) + 1;
            if (bsize < 12 + xlen + 8) return 0;
            *xlen_out = xlen;
            return bsize;
        }
        q += 4 + slen;
    }
    return 0;
}

// Raw inflate of one block's deflate data into exactly `isize` bytes.
bool inflate_block(z_stream& z, const uint8_t* in, size_t n_in, uint8_t* out, uint32_t isize) {
    inflateReset(&z);
    z.next_in = const_cast<Bytef*>(in);
    z.avail_in = (uInt)n_in;
    uint8_t spare;
    z.next_out = isize ? out : &spare;
    z.avail_out = isize ? isize : 0;
    const int r = inflate(&z, Z_FINISH);
    return r == Z_STREAM_END && z.total_out == isize;
}

std::string quoted(const std::string& path) { return "\"" + path + "\""; }

}  // namespace

bool is_bam(const char* path) {
    struct stat sb;
    if (!path || stat(path, &sb) != 0 || !S_ISREG(sb.st_mode)) return false;     // pipes are never opened here (SAM path)
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return false;
    std::vector<uint8_t> b(BGZF_MAX + 8);
    size_t got = 0;
    while (got < b.size()) {
        const ssize_t r = pread(fd, b.data() + got, b.size() - got, (off_t)got);
        if (r <= 0) break;
        got += (size_t)r;
    }
    close(fd);
    uint32_t xlen = 0;
    const uint32_t bs = bgzf_block(b.data(), got, &xlen);
    if (!bs || bs > got) return false;
    z_stream z{};
    if (inflateInit2(&z, -15) != Z_OK) return false;
    uint8_t out[4];
    z.next_in = b.data() + 12 + xlen;
    z.avail_in = bs - 12 - xlen - 8;
    z.next_out = out;
    z.avail_out = 4;
    const int r = inflate(&z, Z_SYNC_FLUSH);
    const bool ok = (r == Z_OK || r == Z_STREAM_END || r == Z_BUF_ERROR) && z.avail_out == 0 && memcmp(out, "BAM\1", 4) == 0;
    inflateEnd(&z);
    return ok;
}

int bam_load(const char* path, const pp_fasta* fa, BamImage& im, std::string& err) {
    using clk = std::chrono::steady_clock;
    const auto t0 = clk::now();
    im = BamImage();
    im.path = path;
    std::string raw;
    if (!read_file(path, raw)) { err = "unable to load alignments from " + quoted(path); return PP_ERR_IO; }
    const auto t1 = clk::now();
    const uint8_t* z = (const uint8_t*)raw.data();
    const size_t zn = raw.size();
    auto bad = [&](const std::string& what) { err = quoted(path) + " is not a valid BAM file: " + what; return PP_ERR_IO; };
    // the BSIZE chain
    struct Blk { uint64_t hdr, at, uoff; uint32_t clen, isize, crc; };
    std::vector<Blk> blocks;
    uint64_t total = 0;
    for (size_t at = 0; at < zn;) {
        uint32_t xlen = 0;
        const uint32_t bs = bgzf_block(z + at, zn - at, &xlen);
        if (!bs) return zn - at < 18 ? bad("truncated BGZF block at byte " + std::to_string(at)) : bad("not BGZF at byte " + std::to_string(at));
        if (bs > zn - at) return bad("truncated BGZF block at byte " + std::to_string(at));
        Blk k;
        k.hdr = at;
        k.at = at + 12 + xlen;
        k.clen = bs - 12 - xlen - 8;
        k.crc = rd32(z + at + bs - 8);
        k.isize = rd32(z + at + bs - 4);
        if (k.isize > BGZF_MAX) return bad("ISIZE mismatch in the BGZF block at byte " + std::to_string(at));
        k.uoff = total;
        total += k.isize;
        blocks.push_back(k);
        at += bs;
    }
    if (blocks.empty() || blocks.back().isize != 0) return bad("no BGZF end-of-file block (the file is truncated)");
    // inflate, one job per block
    im.data.resize_zero(total + PAD);
    {
        const size_t nb = blocks.size();
        const unsigned nt = (unsigned)std::min<size_t>(std::min(16u, std::max(1u, std::thread::hardware_concurrency())), nb / 8 + 1);
        std::vector<uint8_t> st(nb, 0);                                          // 1 ISIZE, 2 CRC32
        std::atomic<size_t> next{0};
        auto work = [&]() {
            z_stream zs{};
            if (inflateInit2(&zs, -15) != Z_OK) { for (auto& s : st) s = 1; return; }
            for (size_t b; (b = next.fetch_add(64)) < nb;)
                for (size_t i = b; i < std::min(nb, b + 64); ++i) {
                    const Blk& k = blocks[i];
                    uint8_t* out = im.data.p + k.uoff;
                    if (!inflate_block(zs, z + k.at, k.clen, out, k.isize)) { st[i] = 1; continue; }
                    if ((uint32_t)crc32(0L, out, k.isize) != k.crc) st[i] = 2;
                }
            inflateEnd(&zs);
        };
        std::vector<std::thread> th;
        for (unsigned t = 1; t < nt; ++t) th.emplace_back(work);
        work();
        for (auto& t : th) t.join();
        for (size_t i = 0; i < nb; ++i)
            if (st[i]) return bad(std::string(st[i] == 1 ? "ISIZE mismatch" : "CRC32 mismatch") + " in the BGZF block at byte " + std::to_string(blocks[i].hdr));
    }
    im.size = total;
    const auto t2 = clk::now();
    // header
    const uint8_t* d = im.data.p;
    if (total < 12 || memcmp(d, "BAM\1", 4) != 0) return bad("no BAM magic");
    const uint64_t l_text = rd32(d + 4);
    if (8 + l_text + 4 > total) return bad("the header runs past the end of the data");
    {
        const char* tx = (const char*)d + 8;
        const size_t tl = strnlen(tx, (size_t)l_text);
        im.header.assign(tx, tl);
    }
    uint64_t p = 8 + l_text;
    const uint32_t n_ref = rd32(d + p);
    p += 4;
    for (uint32_t r = 0; r < n_ref; ++r) {
        if (p + 4 > total) return bad("the header runs past the end of the data");
        const uint64_t l = rd32(d + p);
        if (p + 4 + l + 4 > total) return bad("the header runs past the end of the data");
        const char* nm = (const char*)d + p + 4;
        im.ref_names.emplace_back(nm, strnlen(nm, (size_t)l));
        p += 4 + l + 4;
    }
    // header lines (str::lines), and whether every one of them is a header line of the SAM text
    if (!im.header.empty() && im.header.back() != '\n') im.header += '\n';
    for_each_line(im.header.data(), im.header.size(), [&](std::string_view s) {
        im.header_lines++;
        if (!s.empty() && s[0] != '@') im.device_ok = false;
        return true;
    });
    im.ref_contig.assign((size_t)n_ref + 1, PP_CONTIG_UNKNOWN);
    for (uint32_t r = 0; r <= n_ref; ++r) {
        const std::string& nm = r ? im.ref_names[r - 1] : std::string("*");
        if (nm.find_first_of("\t\r\n") != std::string::npos) im.device_ok = false;
        if (fa) { auto it = fa->index.find(nm); if (it != fa->index.end()) im.ref_contig[r] = it->second; }
    }
    // the block_size chain (records may span BGZF blocks)
    for (uint64_t k = 0; p < total; ++k) {
        if (total - p < 4) return bad("record " + std::to_string(k + 1) + " runs past the end of the data");
        const uint64_t bs = rd32(d + p);
        if (bs < tok::BAM_FIXED - 4) return bad("record " + std::to_string(k + 1) + " runs past its block_size");
        if (total - p - 4 < bs) return bad("record " + std::to_string(k + 1) + " runs past the end of the data");
        im.rec.push_back(p);
        p += 4 + bs;
    }
    const auto t3 = clk::now();
    im.read_ms = std::chrono::duration<float, std::milli>(t1 - t0).count();
    im.inflate_ms = std::chrono::duration<float, std::milli>(t2 - t1).count();
    im.walk_ms = std::chrono::duration<float, std::milli>(t3 - t2).count();
    return PP_OK;
}

namespace {

const char* const FAULT[4] = {"", "runs past its block_size", "has a refID or next_refID out of range", "has malformed optional fields"};

void put_int(std::string& o, int64_t v) { char t[24]; o.append(t, (size_t)snprintf(t, sizeof t, "%lld", (long long)v)); }

// SAM line of record k (its bytes at s).  false: a structural fault (err set).
bool render(const BamImage& im, uint64_t k, std::string& o, std::string& err) {
    tok::Txt x(im.data.p);
    const uint64_t s = im.rec[k];
    tok::BamFix f;
    tok::bam_fixed(x, s, f);
    tok::BamAux a;
    const uint8_t fault = tok::bam_check(x, s, f, (uint32_t)im.ref_names.size(), a);
    if (fault) { err = quoted(im.path) + " is not a valid BAM file: record " + std::to_string(k + 1) + " " + FAULT[fault]; return false; }
    const char* d = (const char*)im.data.p;
    auto ref = [&](int32_t r) -> const std::string& { static const std::string star("*"); return r < 0 ? star : im.ref_names[(size_t)r]; };
    o.append(d + s + tok::BAM_FIXED, f.l_name ? f.l_name - 1 : 0);
    o += '\t'; put_int(o, f.flag);
    o += '\t'; o += ref(f.ref);
    o += '\t'; put_int(o, (int64_t)f.pos + 1);
    o += '\t'; put_int(o, f.mapq);
    o += '\t';
    const uint64_t c0 = s + tok::BAM_FIXED + f.l_name;
    uint64_t cp = c0;
    uint32_t nc = f.n_cigar;
    if (a.cg && tok::bam_placeholder(x, s, f)) { cp = a.cg_pos; nc = a.cg_n; }
    if (nc == 0) o += '*';
    for (uint32_t i = 0; i < nc; ++i) {
        const uint32_t op = rd32(im.data.p + cp + 4ull * i);
        put_int(o, op >> 4);
        o += "MIDNSHP=XB??????"[op & 15];
    }
    o += '\t'; o += f.next_ref == -1 ? std::string("*") : f.next_ref == f.ref ? std::string("=") : ref(f.next_ref);
    o += '\t'; put_int(o, (int64_t)f.next_pos + 1);
    o += '\t'; put_int(o, f.tlen);
    o += '\t';
    if (f.l_seq == 0) o += '*';
    const uint8_t* sq = im.data.p + c0 + 4ull * f.n_cigar;
    for (uint32_t i = 0; i < f.l_seq; ++i) o += "=ACMGRSVTWYHKDBN"[(i & 1) ? (sq[i >> 1] & 15) : (sq[i >> 1] >> 4)];
    o += "\t*";
    // NM and ZP, in their order
    const uint8_t* e = im.data.p + s + 4 + f.block_size;
    for (const uint8_t* q = im.data.p + s + tok::bam_aux_rel(f); q < e;) {
        const uint8_t t0 = q[0], t1 = q[1], ty = q[2];
        q += 3;
        const uint32_t fs = tok::aux_size(ty);
        if (fs) {
            if (t0 == 'N' && t1 == 'M' && tok::is_int_type(ty)) {
                tok::Txt y(im.data.p);
                o += "\tNM:i:";
                put_int(o, tok::aux_int(y, (uint64_t)(q - im.data.p), ty));
            }
            q += fs;
        } else if (ty == 'Z' || ty == 'H') {
            const size_t l = strlen((const char*)q);
            if (ty == 'Z' && tok::lower(t0) == 'z' && tok::lower(t1) == 'p') {
                o += '\t'; o += (char)t0; o += (char)t1; o += ":Z:"; o.append((const char*)q, l);
            }
            q += l + 1;
        } else {                                                         // 'B' (bam_check has validated the layout)
            q += 5 + (uint64_t)rd32(q + 1) * tok::aux_size(q[0]);
        }
    }
    o += '\n';
    return true;
}

}  // namespace

int bam_to_sam(const BamImage& im, std::string& out, std::string& err) {
    const uint64_t n = im.rec.size();
    const unsigned hw = std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
    const unsigned nt = (unsigned)std::min<uint64_t>(hw, n / 20000 + 1);
    std::vector<std::string> part(nt), perr(nt);
    std::vector<uint64_t> bad(nt, ~0ull);
    auto work = [&](unsigned t) {
        const uint64_t lo = n * t / nt, hi = n * (t + 1) / nt;
        std::string& o = part[t];
        o.reserve((size_t)((im.size / std::max<uint64_t>(n, 1)) * (hi - lo) * 2));
        for (uint64_t k = lo; k < hi; ++k)
            if (!render(im, k, o, perr[t])) { bad[t] = k; return; }
    };
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work, t);
    work(0);
    for (auto& t : th) t.join();
    for (unsigned t = 0; t < nt; ++t)
        if (bad[t] != ~0ull) { err = perr[t]; return PP_ERR_IO; }
    size_t total = im.header.size();
    for (auto& p : part) total += p.size();
    out.clear();
    out.reserve(total);
    out += im.header;
    for (auto& p : part) { out += p; std::string().swap(p); }
    return PP_OK;
}

// Cuts before records a BAM's records can be split at for n decoders: cut[0] = 0, cut[n] = the record count, every other cut is
// an aligned record whose QNAME differs from that of the aligned record before it, which is not empty (alignment.rs:255: a
// record joins the open group when the open name is empty or equal; unaligned records never end a group).
void bam_split(const BamImage& im, int n, std::vector<uint64_t>& cut) {
    const uint64_t R = im.rec.size();
    cut.assign((size_t)n + 1, R);
    cut[0] = 0;
    const uint8_t* d = im.data.p;
    auto ok = [&](uint64_t k) {                                    // a record whose fixed part and name are inside its block
        const uint64_t s = im.rec[k];
        return rd32(d + s) >= tok::BAM_FIXED - 4 + (uint32_t)d[s + 12];
    };
    auto aligned = [&](uint64_t k) { return ok(k) && !(rd16(d + im.rec[k] + 18) & 4); };
    auto name = [&](uint64_t k) {
        const uint32_t l = d[im.rec[k] + 12];
        return std::string_view((const char*)d + im.rec[k] + tok::BAM_FIXED, l ? l - 1 : 0);
    };
    for (int g = 1; g < n; ++g) {
        uint64_t k = std::max<uint64_t>(R / (uint64_t)n * (uint64_t)g, cut[g - 1]);
        if (k == 0) k = 1;
        // the last aligned record before k
        int64_t prev = (int64_t)k - 1;
        while (prev >= 0 && !aligned((uint64_t)prev)) --prev;
        for (; k < R; ++k) {
            if (!aligned(k)) continue;
            if (prev >= 0 && !name((uint64_t)prev).empty() && name((uint64_t)prev) != name(k)) break;
            prev = (int64_t)k;
        }
        cut[g] = std::max(k, cut[g - 1]);
    }
}

// ---- writing BAM (the synthetic data sets) -----------------------------------------------------------------------------------

namespace {

// SAMv1 §5.3 reg2bin, 0-based [beg, end)
int reg2bin(int64_t beg, int64_t end) {
    --end;
    if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}

void put32(std::string& o, uint32_t v) { char b[4] = {(char)v, (char)(v >> 8), (char)(v >> 16), (char)(v >> 24)}; o.append(b, 4); }
void put16(std::string& o, uint32_t v) { char b[2] = {(char)v, (char)(v >> 8)}; o.append(b, 2); }

}  // namespace

BgzfWriter::BgzfWriter(const char* path, int level, unsigned threads) : level_(level) {
    f_ = fopen(path, "wb");
    threads_ = threads ? threads : std::max(1u, std::thread::hardware_concurrency());
}

BgzfWriter::~BgzfWriter() { if (f_) fclose(f_); }

// Compresses whole 64 KiB - 256 byte pieces of the buffer in parallel and writes them in order; `all`: the tail as well.
bool BgzfWriter::flush(bool all) {
    constexpr size_t PIECE = BGZF_MAX - 256;
    const size_t n_pieces = all ? (buf_.size() + PIECE - 1) / PIECE : buf_.size() / PIECE;
    if (!f_ || !ok_) return false;
    if (n_pieces == 0) return true;
    std::vector<std::string> out(n_pieces);
    std::atomic<size_t> next{0};
    std::atomic<bool> good{true};
    auto work = [&]() {
        std::vector<uint8_t> tmp(BGZF_MAX + 1024);
        for (size_t i; (i = next.fetch_add(1)) < n_pieces;) {
            const uint8_t* src = (const uint8_t*)buf_.data() + i * PIECE;
            const size_t len = std::min(PIECE, buf_.size() - i * PIECE);
            z_stream z{};
            if (deflateInit2(&z, level_, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) { good = false; return; }
            z.next_in = const_cast<Bytef*>(src);
            z.avail_in = (uInt)len;
            z.next_out = tmp.data();
            z.avail_out = (uInt)tmp.size();
            const int r = deflate(&z, Z_FINISH);
            const size_t clen = z.total_out;
            deflateEnd(&z);
            if (r != Z_STREAM_END || clen + 26 > BGZF_MAX) { good = false; return; }
            std::string& o = out[i];
            static const uint8_t hdr[12] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0};
            o.append((const char*)hdr, 12);
            o += "BC"; put16(o, 2); put16(o, (uint32_t)(clen + 25));
            o.append((const char*)tmp.data(), clen);
            put32(o, (uint32_t)crc32(0L, src, (uInt)len));
            put32(o, (uint32_t)len);
        }
    };
    std::vector<std::thread> th;
    const unsigned nt = (unsigned)std::min<size_t>(threads_, n_pieces);
    for (unsigned t = 1; t < nt; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
    if (!good) return ok_ = false;
    for (auto& o : out)
        if (fwrite(o.data(), 1, o.size(), f_) != o.size()) return ok_ = false;
    buf_.erase(0, std::min(buf_.size(), n_pieces * PIECE));
    return true;
}

bool BgzfWriter::write(const void* p, size_t n) {
    buf_.append((const char*)p, n);
    return buf_.size() < (16u << 20) || flush(false);
}

bool BgzfWriter::close() {
    if (!f_) return false;
    bool good = flush(true);
    static const uint8_t eof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    good = good && fwrite(eof, 1, 28, f_) == 28;
    good = (fclose(f_) == 0) && good;
    f_ = nullptr;
    return good && ok_;
}

void bam_header(const std::string& text, const std::vector<std::pair<std::string, uint64_t>>& refs, std::string& o) {
    o += "BAM\1";
    put32(o, (uint32_t)text.size());
    o += text;
    put32(o, (uint32_t)refs.size());
    for (auto& r : refs) {
        put32(o, (uint32_t)r.first.size() + 1);
        o += r.first; o += '\0';
        put32(o, (uint32_t)r.second);
    }
}

// One SAM line (no newline) of the synthetic generator -> one BAM record: the eleven columns, and every optional field of
// type i (stored in the smallest integer type that holds it, as samtools does) or Z.  false: not a line of that shape.
bool sam_line_to_bam(std::string_view s, const std::unordered_map<std::string, int32_t>& ref_id, std::string& o) {
    std::string_view f[11];
    size_t pos = 0;
    for (int k = 0; k < 11; ++k) {
        const size_t t = s.find('\t', pos);
        if (t == std::string_view::npos && k < 10) return false;
        f[k] = s.substr(pos, (t == std::string_view::npos ? s.size() : t) - pos);
        pos = t == std::string_view::npos ? s.size() + 1 : t + 1;
    }
    auto num = [](std::string_view v) { return (int64_t)strtoll(std::string(v).c_str(), nullptr, 10); };
    auto rid = [&](std::string_view v, int32_t self) -> int32_t {
        if (v == "*") return -1;
        if (v == "=") return self;
        auto it = ref_id.find(std::string(v));
        return it == ref_id.end() ? -2 : it->second;
    };
    const int32_t ref = rid(f[2], -1);
    const int32_t nref = rid(f[6], ref);
    if (ref < -1 || nref < -1) return false;
    std::vector<uint32_t> cig;
    int64_t rlen = 0;
    if (f[5] != "*") {
        uint64_t len = 0;
        for (char c : f[5]) {
            if (c >= '0' && c <= '9') { len = len * 10 + (uint64_t)(c - '0'); continue; }
            const char* L = strchr("MIDNSHP=X", c);
            if (!L || !c) return false;
            const uint32_t op = (uint32_t)(L - "MIDNSHP=X");
            cig.push_back((uint32_t)(len << 4) | op);
            if (op == PP_OP_M || op == PP_OP_D || op == PP_OP_N || op == PP_OP_EQ || op == PP_OP_X) rlen += (int64_t)len;
            len = 0;
        }
    }
    const std::string_view seq = f[9] == "*" ? std::string_view() : f[9];
    const int64_t pos0 = num(f[3]) - 1;
    const size_t at = o.size();
    put32(o, 0);                                                       // block_size, set below
    put32(o, (uint32_t)ref);
    put32(o, (uint32_t)(int32_t)pos0);
    o += (char)(f[0].size() + 1);
    o += (char)(uint8_t)num(f[4]);
    put16(o, (uint32_t)reg2bin(pos0 < 0 ? 0 : pos0, (pos0 < 0 ? 0 : pos0) + std::max<int64_t>(rlen, 1)));
    put16(o, (uint32_t)cig.size());
    put16(o, (uint32_t)num(f[1]));
    put32(o, (uint32_t)seq.size());
    put32(o, (uint32_t)nref);
    put32(o, (uint32_t)(int32_t)(num(f[7]) - 1));
    put32(o, (uint32_t)(int32_t)num(f[8]));
    o += f[0]; o += '\0';
    for (uint32_t c : cig) put32(o, c);
    static const std::string codes = "=ACMGRSVTWYHKDBN";
    for (size_t i = 0; i < seq.size(); i += 2) {
        auto code = [&](char c) { const size_t k = codes.find((char)(c >= 'a' && c <= 'z' ? c - 32 : c)); return k == std::string::npos ? 15u : (uint32_t)k; };
        o += (char)((code(seq[i]) << 4) | (i + 1 < seq.size() ? code(seq[i + 1]) : 0u));
    }
    if (f[10] == "*") o.append(seq.size(), (char)0xff);
    else for (char c : f[10]) o += (char)(c - 33);
    while (pos <= s.size()) {
        const size_t t = s.find('\t', pos);
        const std::string_view tag = s.substr(pos, (t == std::string_view::npos ? s.size() : t) - pos);
        pos = t == std::string_view::npos ? s.size() + 1 : t + 1;
        if (tag.size() < 5 || tag[2] != ':' || tag[4] != ':') return false;
        o.append(tag.data(), 2);
        const std::string_view v = tag.substr(5);
        if (tag[3] == 'i') {
            const int64_t x = num(v);
            if (x >= 0 && x <= 255) { o += 'C'; o += (char)x; }
            else if (x >= -128 && x <= 127) { o += 'c'; o += (char)x; }
            else if (x >= 0 && x <= 65535) { o += 'S'; put16(o, (uint32_t)x); }
            else if (x >= -32768 && x <= 32767) { o += 's'; put16(o, (uint32_t)x); }
            else if (x >= 0) { o += 'I'; put32(o, (uint32_t)x); }
            else { o += 'i'; put32(o, (uint32_t)x); }
        } else if (tag[3] == 'Z') {
            o += 'Z'; o += v; o += '\0';
        } else {
            return false;
        }
    }
    const uint32_t bs = (uint32_t)(o.size() - at - 4);
    memcpy(&o[at], &bs, 4);
    return true;
}

}  // namespace pp
