// sam_pack.cpp — SAM text -> packed struct-of-arrays alignments (pp_alignments) for the polish path.
//
// Host side of the boundary: restates the TEXT handling of the reference, nothing else.
//   add_to_pileup   /root/reference/src/alignment.rs:225-272  (line loop, '@'/empty skipping, grouping)
//   Alignment::new  /root/reference/src/alignment.rs:49-98    (columns, FLAG/POS, NM / ZP tags, CIGAR check)
//   get_expanded_cigar :325-346 (validation only: the CIGAR is kept run-length encoded, never expanded)
//   get_read_seq_from_alignments :311-322 and add_read_seq :161-167 (source sequence of SEQ="*" records)
// Everything downstream (goodness, k, CIGAR walk, trim, pileup, vote) happens on the device.
#include <algorithm>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <cstdio>
#include <cstdlib>
#include <thread>

#include "pp_internal.h"

namespace {

struct NibTable {
    uint8_t t[256];
    NibTable() {
        memset(t, 0, sizeof t);
        const char* codes = "=ACMGRSVTWYHKDBN";
        for (int i = 1; i < 16; ++i) {
            t[(unsigned char)codes[i]] = (uint8_t)i;
            t[(unsigned char)(codes[i] + 32)] = (uint8_t)i;  // lower case: SEQ is upper-cased (alignment.rs:94)
        }
    }
};
const NibTable NIB;

inline int op_code(char c) {
    switch (c) {
        case 'M': return PP_OP_M; case 'I': return PP_OP_I; case 'D': return PP_OP_D; case 'N': return PP_OP_N;
        case 'S': return PP_OP_S; case 'H': return PP_OP_H; case 'P': return PP_OP_P; case '=': return PP_OP_EQ;
        case 'X': return PP_OP_X; default: return -1;
    }
}

inline bool eq_ignore_case(std::string_view a, const char* b, size_t n) {
    if (a.size() != n) return false;
    for (size_t i = 0; i < n; ++i) {
        char x = a[i], y = b[i];
        if (x >= 'A' && x <= 'Z') x = (char)(x + 32);
        if (y >= 'A' && y <= 'Z') y = (char)(y + 32);
        if (x != y) return false;
    }
    return true;
}

std::string rust_debug_str(std::string_view s) {  // {:?} of a str, common escapes only
    std::string o = "\"";
    for (char c : s) {
        if (c == '"') o += "\\\""; else if (c == '\\') o += "\\\\"; else if (c == '\t') o += "\\t"; else o += c;
    }
    return o + "\"";
}

struct GroupState {
    bool name_empty = true;          // current_read_name.is_empty() (alignment.rs:255)
    std::string_view name;
    uint64_t first_aln = 0, n = 0;   // alignments of the open group
    bool have_src = false;
    uint64_t src_aln = 0;            // first record of the group whose SEQ is not "*" (alignment.rs:311-318)
};

// Closes a read group (process_one_read's text side, alignment.rs:275-295): read id, and for SEQ="*" records the group's
// source sequence (copy or reverse complement by strand).  Returns false on the reference's "no sequence" error.
bool finalize_group(pp_pack* P, const GroupState& g, std::string& err) {
    const uint64_t gid = P->group_name_off.size();
    if (gid >= 0xFFFFFFFFull) { err = "more than 2^32-1 reads in one call are not supported"; return false; }
    P->group_name_off.push_back(P->name_pool.size());
    P->name_pool.append(g.name.data(), g.name.size());
    P->name_pool.push_back('\0');
    const bool skipped = P->careful && g.n > 1;   // alignment.rs:277-279
    if (!g.have_src && !skipped) { err = "no alignments for read " + std::string(g.name) + " contain sequence"; return false; }
    const uint32_t src_off = g.have_src ? P->seq_off[g.src_aln] : 0;
    const uint16_t src_len = g.have_src ? P->seq_len[g.src_aln] : 0;
    const uint8_t src_rev = g.have_src ? (P->flags[g.src_aln] & PP_FLAG_REVERSE) : 0;
    for (uint64_t a = g.first_aln; a < g.first_aln + g.n; ++a) {
        P->read_id[a] = (uint32_t)gid;
        if (P->flags[a] & PP_FLAG_SEQSTAR) {
            if (g.have_src) {
                P->seq_off[a] = src_off;
                P->seq_len[a] = src_len;
                if ((P->flags[a] & PP_FLAG_REVERSE) != src_rev) P->flags[a] |= PP_FLAG_RC;
            } else {
                P->flags[a] |= PP_FLAG_NOSEQ;
            }
        }
    }
    return true;
}

struct DeferredGroup { std::string_view name; uint64_t first, n; bool have_src; uint64_t src_aln; };

struct Packer {
    pp_pack* P;
    const std::string& fname;
    GroupState g;
    uint64_t line_count = 0, alignment_count = 0, read_count = 0;
    std::vector<DeferredGroup>* deferred = nullptr;   // chunk mode: groups are only recorded; the merge closes them

    bool fail(int code, const std::string& m) { P->error = m; P->error_code = code; return false; }

    bool close_group() {
        if (g.n == 0) return true;
        if (deferred) {
            deferred->push_back({g.name, g.first_aln, g.n, g.have_src, g.src_aln});
        } else {
            read_count++;
            std::string err;
            if (!finalize_group(P, g, err)) return fail(PP_ERR_INPUT, err);
        }
        g.n = 0;
        g.have_src = false;
        return true;
    }

    // Stores one sequence in the pool; returns false on unsupported input.
    bool store_seq(std::string_view seq, uint32_t& off) {
        if (P->seq_blocks >= 0xFFFFFFFFull) return fail(PP_ERR_INPUT, "sequence pool exceeds 2^32 blocks");
        off = (uint32_t)P->seq_blocks;
        size_t len = seq.size();
        size_t blocks = (len + PP_SEQ_BLOCK - 1) / PP_SEQ_BLOCK;
        if (P->seq_bits == 4) {
            size_t base = P->seq_blocks * (PP_SEQ_BLOCK / 2);
            P->seq_pool.resize_zero(base + blocks * (PP_SEQ_BLOCK / 2));
            uint8_t* d = P->seq_pool.p + base;
            bool exotic = false;
            for (size_t j = 0; j < len; ++j) {
                uint8_t c = NIB.t[(unsigned char)seq[j]];
                exotic |= (c == 0);
                d[j >> 1] |= (uint8_t)(c << ((j & 1) * 4));
            }
            if (exotic) P->need8 = true;
        } else {
            size_t base = P->seq_blocks * PP_SEQ_BLOCK;
            P->seq_pool.resize_zero(base + blocks * PP_SEQ_BLOCK);
            uint8_t* d = P->seq_pool.p + base;
            for (size_t j = 0; j < len; ++j) {
                char c = seq[j];
                d[j] = (uint8_t)((c >= 'a' && c <= 'z') ? c - 32 : c);
            }
        }
        P->seq_blocks += blocks;
        return true;
    }

    bool line(std::string_view s) {
        line_count++;
        if (s.empty() || s[0] == '@') return true;     // alignment.rs:241-242
        // split('\t'): need fields 0,1,2,3,5,9 and everything from 11 on
        std::string_view f[11];
        size_t pos = 0, nf = 0;
        while (nf < 11) {
            const char* t = (const char*)memchr(s.data() + pos, '\t', s.size() - pos);
            if (!t) { f[nf++] = s.substr(pos); pos = s.size() + 1; break; }
            size_t e = (size_t)(t - s.data());
            f[nf++] = s.substr(pos, e - pos);
            pos = e + 1;
        }
        auto where = [&]() { return " in \"" + fname + "\" (line " + std::to_string(line_count) + ")"; };
        if (nf < 11) return fail(PP_ERR_INPUT, "too few columns" + where());
        uint64_t v;
        if (!pp::parse_uint(f[1], 0xFFFFFFFFull, v)) return fail(PP_ERR_INPUT, "invalid FLAG field " + rust_debug_str(f[1]) + where());
        uint32_t sam_flags = (uint32_t)v;
        if (!pp::parse_uint(f[3], ~0ull, v)) return fail(PP_ERR_INPUT, "invalid POS field " + rust_debug_str(f[3]) + where());
        uint64_t rstart = v > 0 ? v - 1 : 0;            // alignment.rs:58-61
        std::string_view cigar = f[5], seq = f[9];

        uint32_t mismatches = 0xFFFFFFFFu;
        bool pass_qc = true;
        while (pos <= s.size()) {                        // tags, alignment.rs:67-75
            const char* t = (const char*)memchr(s.data() + pos, '\t', s.size() - pos);
            size_t e = t ? (size_t)(t - s.data()) : s.size();
            std::string_view p = s.substr(pos, e - pos);
            if (p.size() >= 5 && memcmp(p.data(), "NM:i:", 5) == 0) {
                if (!pp::parse_uint(p.substr(5), 0xFFFFFFFFull, v)) return fail(PP_ERR_INPUT, "invalid NM tag " + rust_debug_str(p) + where());
                mismatches = (uint32_t)v;
            }
            if (eq_ignore_case(p, "ZP:Z:fail", 9)) pass_qc = false;
            pos = e + 1;
        }
        bool aligned = (sam_flags & 4) == 0;
        if (mismatches == 0xFFFFFFFFu && aligned) return fail(PP_ERR_INPUT, "missing NM tag" + where());

        // CIGAR: must be "*" or a concatenation of \d+[MIDNSHP=X] tokens (alignment.rs:325-346)
        size_t ops_begin = P->cigar_ops.size();
        bool cigar_ok = true;
        if (!(cigar.size() == 1 && cigar[0] == '*')) {
            size_t i = 0, n = cigar.size();
            while (i < n) {
                uint64_t len = 0;
                size_t j = i;
                bool big = false;
                while (j < n && cigar[j] >= '0' && cigar[j] <= '9') {
                    len = len * 10 + (uint64_t)(cigar[j] - '0');
                    if (len > 0xFFFFFFFFull) big = true;
                    j++;
                }
                int op = (j < n && j > i) ? op_code(cigar[j]) : -1;
                if (op < 0) { cigar_ok = false; break; }
                if (big) { P->cigar_ops.resize(ops_begin); return fail(PP_ERR_INPUT, "CIGAR operation length does not fit u32 for read " + std::string(f[0])); }
                if (len > 0 && aligned) {
                    if (len >= (1ull << 28)) { P->cigar_ops.resize(ops_begin); return fail(PP_ERR_INPUT, "CIGAR operation longer than 2^28-1 is not supported (read " + std::string(f[0]) + ")"); }
                    P->cigar_ops.push_back((uint32_t)(len << 4) | (uint32_t)op);
                }
                i = j + 1;
            }
        }
        if (!cigar_ok) {
            P->cigar_ops.resize(ops_begin);
            return fail(PP_ERR_INPUT, "encountered an invalid CIGAR string for read " + std::string(f[0]) + ": " + rust_debug_str(cigar));
        }
        if (!aligned) { P->cigar_ops.resize(ops_begin); return true; }   // alignment.rs:250

        alignment_count++;
        size_t nops = P->cigar_ops.size() - ops_begin;
        if (nops == 0)   // the reference panics in starts_and_ends_with_match (alignment.rs:156)
            return fail(PP_ERR_INPUT, "aligned record of read " + std::string(f[0]) + " has an empty CIGAR" + where());
        if (nops > 0xFFFF) return fail(PP_ERR_INPUT, "more than 65535 CIGAR operations in one record are not supported" + where());
        if (ops_begin > 0xFFFFFFFFull) return fail(PP_ERR_INPUT, "CIGAR pool exceeds 2^32 operations");
        if (rstart > 0xFFFFFFFEull) return fail(PP_ERR_INPUT, "alignment start beyond 2^32 is not supported" + where());

        // grouping (alignment.rs:255-263)
        std::string_view name = f[0];
        if (!(g.name_empty || g.name == name)) {
            if (!close_group()) return false;
        }
        if (g.n == 0) g.first_aln = P->contig.size();
        g.name = name;
        g.name_empty = name.empty();
        g.n++;

        uint32_t cidx = PP_CONTIG_UNKNOWN;
        {
            P->tmp.assign(f[2].data(), f[2].size());
            auto it = P->fasta->index.find(P->tmp);
            if (it != P->fasta->index.end()) cidx = it->second;
            else P->unknown_ref.emplace(P->contig.size(), P->tmp);
        }
        uint8_t fl = 0;
        if (sam_flags & 16) fl |= PP_FLAG_REVERSE;
        if (!pass_qc) fl |= PP_FLAG_ZPFAIL;
        uint32_t soff = 0;
        uint16_t slen = 0;
        if (seq.size() == 1 && seq[0] == '*') {
            fl |= PP_FLAG_SEQSTAR;
        } else {
            if (seq.size() > 0xFFFF) return fail(PP_ERR_INPUT, "reads longer than 65535 bases are not supported" + where());
            if (!store_seq(seq, soff)) return false;
            slen = (uint16_t)seq.size();
            if (!g.have_src) {                          // first record whose SEQ != "*" (alignment.rs:311-318)
                g.have_src = true;
                g.src_aln = P->contig.size();
            }
        }
        P->contig.push_back(cidx);
        P->ref_start.push_back((uint32_t)rstart);
        P->read_id.push_back(0);
        P->seq_off.push_back(soff);
        P->seq_len.push_back(slen);
        P->cigar_off.push_back((uint32_t)ops_begin);
        P->n_cigar.push_back((uint16_t)nops);
        P->nm.push_back(mismatches);
        P->flags.push_back(fl);
        return true;
    }
};

int finish_file(pp_pack* P, Packer& pk, const std::string& fname) {
    if (pk.alignment_count == 0) {     // alignment.rs:268-270
        P->error = "no alignments in \"" + fname + "\"";
        P->error_code = PP_ERR_INPUT;
        return PP_ERR_INPUT;
    }
    if (!pk.close_group()) return P->error_code;
    pp_pack::FileStat st;
    st.name = fname;
    st.alignments = pk.alignment_count;
    st.reads = pk.read_count;
    P->files.push_back(st);
    return PP_OK;
}

int pack_text(pp_pack* P, const char* data, size_t n, const std::string& fname) {
    Packer pk{P, fname};
    bool ok = true;
    pp::for_each_line(data, n, [&](std::string_view s) { ok = pk.line(s); return ok; });
    if (!ok) return P->error_code;
    return finish_file(P, pk, fname);
}

// Streaming variant: one logical SAM file fed in chunks of whole lines.  The QNAME of the open group must
// outlive a chunk, so it is copied.
struct Stream {
    std::string fname;
    Packer pk;
    std::string open_name;
    Stream(pp_pack* P, const char* n) : fname(n ? n : "<stream>"), pk{P, fname} {}
};

void clear_arrays(pp_pack* P) {
    P->contig.clear(); P->ref_start.clear(); P->read_id.clear(); P->seq_off.clear(); P->cigar_off.clear();
    P->nm.clear(); P->seq_len.clear(); P->n_cigar.clear(); P->flags.clear(); P->cigar_ops.clear();
    P->seq_pool.clear(); P->seq_blocks = 0; P->name_pool.clear(); P->group_name_off.clear();
    P->unknown_ref.clear(); P->files.clear();
}


// ---- parallel parse of one SAM file -----------------------------------------------------------------------------
// The text is cut into chunks at line starts; each chunk is parsed by its own thread into private arrays with its
// read groups only RECORDED; the merge then walks the chunks in file order, appends their arrays (rebasing pool
// offsets), re-applies the reference's grouping rule across every chunk seam (a group continues into the next chunk iff
// the open name is empty or equals the next record's QNAME, alignment.rs:255) and closes the groups exactly as the
// sequential path does.  Errors keep file order: the first chunk with a text error ends the file there.
struct ChunkOut {
    pp_pack tmp;
    std::vector<DeferredGroup> groups;
    uint64_t first_line = 0, n_lines = 0, alignments = 0;
    bool ok = true;
};

uint64_t count_lines(const char* p, size_t n) {
    uint64_t c = 0;
    const char* e = p + n;
    while (p < e) { const char* q = (const char*)memchr(p, '\n', (size_t)(e - p)); if (!q) { c++; break; } c++; p = q + 1; }
    return c;
}

template <class T> void append_vec(std::vector<T>& dst, const std::vector<T>& src) { dst.insert(dst.end(), src.begin(), src.end()); }

int pack_text_parallel(pp_pack* P, const char* data, size_t n, const std::string& fname, unsigned n_threads, size_t min_chunk) {
    // chunk boundaries at line starts
    std::vector<size_t> cut{0};
    const size_t want = std::max(min_chunk, n / n_threads + 1);
    while (cut.back() < n) {
        size_t nxt = cut.back() + want;
        if (nxt >= n) { cut.push_back(n); break; }
        const char* q = (const char*)memchr(data + nxt, '\n', n - nxt);
        cut.push_back(q ? (size_t)(q - data) + 1 : n);
    }
    const size_t nc = cut.size() - 1;
    std::vector<ChunkOut> out(nc);
    {   // line numbers of chunk starts (error messages carry file line numbers)
        std::vector<std::thread> th;
        for (size_t c = 0; c < nc; ++c) th.emplace_back([&, c] { out[c].n_lines = count_lines(data + cut[c], cut[c + 1] - cut[c]); });
        for (auto& t : th) t.join();
        uint64_t base = 0;
        for (size_t c = 0; c < nc; ++c) { out[c].first_line = base; base += out[c].n_lines; }
    }
    {
        std::vector<std::thread> th;
        for (size_t c = 0; c < nc; ++c) th.emplace_back([&, c] {
            ChunkOut& o = out[c];
            o.tmp.fasta = P->fasta; o.tmp.careful = P->careful; o.tmp.seq_bits = P->seq_bits;
            {   // every array sized once from the chunk's line count: growing them by reallocation means mmap / munmap calls that
                // serialise the threads on the process's address-space lock (measured: 8 threads no faster than one)
                pp_pack& t = o.tmp;
                const size_t nl = (size_t)o.n_lines + 1, bytes = cut[c + 1] - cut[c];
                t.contig.reserve(nl); t.ref_start.reserve(nl); t.read_id.reserve(nl); t.seq_off.reserve(nl); t.cigar_off.reserve(nl);
                t.nm.reserve(nl); t.seq_len.reserve(nl); t.n_cigar.reserve(nl); t.flags.reserve(nl);
                t.cigar_ops.reserve(nl + nl / 2);
                t.seq_pool.reserve((t.seq_bits == 4 ? bytes / 2 : bytes) + 32 * nl);     // an upper bound; untouched pages cost nothing
                o.groups.reserve(nl / 2 + 1);
            }
            Packer pk{&o.tmp, fname};
            pk.deferred = &o.groups;
            pk.line_count = o.first_line;
            bool ok = true;
            pp::for_each_line(data + cut[c], cut[c + 1] - cut[c], [&](std::string_view s) { ok = pk.line(s); return ok; });
            if (ok) pk.close_group();              // records the chunk's last (possibly still open) group
            o.ok = ok;
            o.alignments = pk.alignment_count;
        });
        for (auto& t : th) t.join();
    }
    // merge in file order
    GroupState carry;                              // the open group of the stream so far
    uint64_t reads = 0, alignments = 0;
    {   // the destination arrays grow once, to the sum of the chunks
        size_t na = P->contig.size(), no = P->cigar_ops.size(), nb = P->seq_pool.n, ng = 0;
        for (size_t c = 0; c < nc; ++c) { na += out[c].tmp.contig.size(); no += out[c].tmp.cigar_ops.size(); nb += out[c].tmp.seq_pool.n; ng += out[c].groups.size(); }
        P->contig.reserve(na); P->ref_start.reserve(na); P->read_id.reserve(na); P->seq_off.reserve(na); P->cigar_off.reserve(na);
        P->nm.reserve(na); P->seq_len.reserve(na); P->n_cigar.reserve(na); P->flags.reserve(na);
        P->cigar_ops.reserve(no);
        P->seq_pool.reserve(nb + 64);
        P->group_name_off.reserve(P->group_name_off.size() + ng);
    }
    auto close_carry = [&]() -> bool {
        if (carry.n == 0) return true;
        reads++;
        std::string err;
        if (!finalize_group(P, carry, err)) { P->error = err; P->error_code = PP_ERR_INPUT; return false; }
        carry.n = 0; carry.have_src = false;
        return true;
    };
    for (size_t c = 0; c < nc; ++c) {
        ChunkOut& o = out[c];
        pp_pack& t = o.tmp;
        const uint64_t aln_base = P->contig.size(), cig_base = P->cigar_ops.size(), blk_base = P->seq_blocks;
        if (cig_base + t.cigar_ops.size() > 0xFFFFFFFFull) { P->error = "CIGAR pool exceeds 2^32 operations"; P->error_code = PP_ERR_INPUT; return PP_ERR_INPUT; }
        if (blk_base + t.seq_blocks > 0xFFFFFFFFull) { P->error = "sequence pool exceeds 2^32 blocks"; P->error_code = PP_ERR_INPUT; return PP_ERR_INPUT; }
        append_vec(P->contig, t.contig); append_vec(P->ref_start, t.ref_start); append_vec(P->read_id, t.read_id);
        append_vec(P->seq_len, t.seq_len); append_vec(P->n_cigar, t.n_cigar); append_vec(P->nm, t.nm); append_vec(P->flags, t.flags);
        append_vec(P->cigar_ops, t.cigar_ops);
        const size_t a0 = P->seq_off.size();
        append_vec(P->seq_off, t.seq_off); append_vec(P->cigar_off, t.cigar_off);
        for (size_t a = a0; a < P->seq_off.size(); ++a) {
            P->cigar_off[a] += (uint32_t)cig_base;
            if (!(P->flags[a] & PP_FLAG_SEQSTAR)) P->seq_off[a] += (uint32_t)blk_base;
        }
        const size_t pool0 = P->seq_pool.n;
        P->seq_pool.resize_zero(pool0 + t.seq_pool.n);
        if (t.seq_pool.n) memcpy(P->seq_pool.p + pool0, t.seq_pool.p, t.seq_pool.n);
        P->seq_blocks += t.seq_blocks;
        for (auto& kv : t.unknown_ref) P->unknown_ref.emplace(kv.first + aln_base, kv.second);
        if (t.need8) P->need8 = true;
        alignments += o.alignments;
        for (size_t gi = 0; gi < o.groups.size(); ++gi) {
            const DeferredGroup& dg = o.groups[gi];
            const bool joins = carry.n > 0 && gi == 0 && (carry.name_empty || carry.name == dg.name);   // alignment.rs:255
            if (!joins && !close_carry()) return P->error_code;
            if (carry.n == 0) { carry.first_aln = dg.first + aln_base; carry.have_src = false; }
            // (a joined group is contiguous: chunk arrays are appended back to back)
            if (!carry.have_src && dg.have_src) { carry.have_src = true; carry.src_aln = dg.src_aln + aln_base; }
            carry.n += dg.n;
            carry.name = dg.name;
            carry.name_empty = dg.name.empty();
            // inside a chunk every recorded group but the last is already complete
            if (gi + 1 < o.groups.size() && !close_carry()) return P->error_code;
        }
        if (!o.ok) { P->error = t.error; P->error_code = t.error_code; return P->error_code; }
    }
    if (alignments == 0) {     // alignment.rs:268-270
        P->error = "no alignments in \"" + fname + "\"";
        P->error_code = PP_ERR_INPUT;
        return PP_ERR_INPUT;
    }
    if (!close_carry()) return P->error_code;
    pp_pack::FileStat st;
    st.name = fname;
    st.alignments = alignments;
    st.reads = reads;
    P->files.push_back(st);
    return PP_OK;
}

}  // namespace

extern "C" pp_pack* pp_pack_create(const pp_fasta* f, int careful) {
    if (!f) return nullptr;
    pp_pack* P = new pp_pack();
    P->fasta = f;
    P->careful = careful != 0;
    return P;
}

extern "C" void pp_pack_free(pp_pack* p) { delete p; }

extern "C" int pp_pack_add_sam_file(pp_pack* P, const char* path) {
    if (!P || !path) return PP_ERR_ARG;
    if (pp::is_bam(path)) {
        // A BAM file is parsed as its SAM text: the header text, then one line per record (bam.cpp), so that every rule and every
        // message of the text path - line numbers included - holds for it unchanged.
        std::string sam, err;
        int rc = PP_OK;
        {
            pp::BamImage im;
            rc = pp::bam_load(path, nullptr, im, err);
            if (rc == PP_OK) rc = pp::bam_to_sam(im, sam, err);
        }
        if (rc != PP_OK) { P->error = err; P->error_code = rc; return rc; }
        if (!P->replaying) P->sources.push_back({true, path, std::string()});
        unsigned nt = P->threads ? P->threads : std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
        return (nt > 1 && sam.size() >= 2 * P->min_chunk) ? pack_text_parallel(P, sam.data(), sam.size(), path, nt, P->min_chunk)
                                                          : pack_text(P, sam.data(), sam.size(), path);
    }
    // A big regular file is read by several threads, each pread()ing its slice straight into one buffer (one pass, the page faults of
    // the buffer spread over the threads); anything else - a small file, a pipe, a device - is read into a string.  (Not mmap: a
    // file that another process truncates while it is parsed would raise SIGBUS; a short read is simply handled.)
    std::string data;
    pp::AlignedBytes big;
    const char* text = nullptr;
    size_t len = 0;
    {
        struct stat sb;                                   // (stat first: a FIFO must be opened exactly once, by read_file below)
        const unsigned rt = std::min(8u, std::max(1u, std::thread::hardware_concurrency()));
        if (stat(path, &sb) == 0 && S_ISREG(sb.st_mode) && (uint64_t)sb.st_size >= (32ull << 20) && rt > 1) {
            const int fd = open(path, O_RDONLY);
            if (fd >= 0) {
                const size_t size = (size_t)sb.st_size;
                big.reserve(size + 64);
                std::vector<char> whole(rt, 0);
                std::vector<std::thread> th;
                for (unsigned t = 0; t < rt; ++t) th.emplace_back([&, t] {
                    size_t at = size * t / rt;
                    const size_t end = size * (t + 1) / rt;
                    while (at < end) {
                        const ssize_t r = pread(fd, big.p + at, end - at, (off_t)at);
                        if (r <= 0) return;                     // shorter than stat said (or an error): the sequential reader decides
                        at += (size_t)r;
                    }
                    whole[t] = 1;
                });
                for (auto& t : th) t.join();
                close(fd);
                if (std::all_of(whole.begin(), whole.end(), [](char c) { return c != 0; })) { big.n = size; text = (const char*)big.p; len = size; }
            }
        }
    }
    if (!text) {
        if (!pp::read_file(path, data)) {
            P->error = std::string("unable to load alignments from \"") + path + "\"";   // alignment.rs:219
            P->error_code = PP_ERR_IO;
            return PP_ERR_IO;
        }
        text = data.data(); len = data.size();
    }
    if (!P->replaying) P->sources.push_back({true, path, std::string()});
    unsigned nt = P->threads ? P->threads : std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
    return (nt > 1 && len >= 2 * P->min_chunk) ? pack_text_parallel(P, text, len, path, nt, P->min_chunk) : pack_text(P, text, len, path);
}

// Parsing threads for pp_pack_add_sam_file (0 = one per hardware thread, at most 16) and the smallest chunk a thread gets.
extern "C" int pp_pack_set_threads(pp_pack* P, uint32_t n_threads, uint64_t min_chunk_bytes) {
    if (!P) return PP_ERR_ARG;
    P->threads = n_threads;
    P->min_chunk = min_chunk_bytes ? (size_t)min_chunk_bytes : (size_t)(8u << 20);
    return PP_OK;
}

extern "C" int pp_pack_add_sam_text(pp_pack* P, const char* text, size_t len, const char* name_for_errors) {
    if (!P || (!text && len)) return PP_ERR_ARG;
    std::string nm = name_for_errors ? name_for_errors : "<memory>";
    if (!P->replaying) P->sources.push_back({false, nm, std::string(text, len)});
    return pack_text(P, text, len, nm);
}

extern "C" int pp_pack_stream_begin(pp_pack* P, const char* name_for_errors) {
    if (!P || P->stream) return PP_ERR_ARG;
    P->stream = new Stream(P, name_for_errors);
    P->no_replay = true;                      // streamed text is not retained: an exotic SEQ byte is an error
    return PP_OK;
}

extern "C" int pp_pack_stream_feed(pp_pack* P, const char* text, size_t len) {
    if (!P || !P->stream) return PP_ERR_ARG;
    Stream* S = (Stream*)P->stream;
    bool ok = true;
    pp::for_each_line(text, len, [&](std::string_view s) { ok = S->pk.line(s); return ok; });
    if (!ok) return P->error_code;
    // keep the open group's QNAME alive beyond this chunk
    S->open_name.assign(S->pk.g.name.data(), S->pk.g.name.size());
    S->pk.g.name = S->open_name;
    return PP_OK;
}

extern "C" int pp_pack_stream_end(pp_pack* P) {
    if (!P || !P->stream) return PP_ERR_ARG;
    Stream* S = (Stream*)P->stream;
    int rc = finish_file(P, S->pk, S->fname);
    delete S;
    P->stream = nullptr;
    return rc;
}

extern "C" int pp_pack_finish(pp_pack* P, pp_alignments* out) {
    if (!P || !out) return PP_ERR_ARG;
    if (P->need8 && P->seq_bits == 4 && P->no_replay) {
        P->error = "a streamed SAM contains a SEQ character outside ACMGRSVTWYHKDBN; feed it as a file or whole text";
        P->error_code = PP_ERR_INPUT;
        return PP_ERR_INPUT;
    }
    if (P->need8 && P->seq_bits == 4) {
        // A read contains a character outside "ACMGRSVTWYHKDBN": repack everything with 8-bit sequences so
        // that allele strings stay byte-exact (pileup.rs:62 counts arbitrary strings).
        clear_arrays(P);
        P->seq_bits = 8;
        P->need8 = false;
        P->replaying = true;
        for (auto& s : P->sources) {
            int rc = s.is_file ? pp_pack_add_sam_file(P, s.path_or_name.c_str())
                               : pp_pack_add_sam_text(P, s.text.data(), s.text.size(), s.path_or_name.c_str());
            if (rc != PP_OK) { P->replaying = false; return rc; }
        }
        P->replaying = false;
    }
    memset(out, 0, sizeof *out);
    out->n_aln = P->contig.size();
    out->n_reads = P->group_name_off.size();
    out->contig = P->contig.data();
    out->ref_start = P->ref_start.data();
    out->read_id = P->read_id.data();
    out->seq_off = P->seq_off.data();
    out->seq_len = P->seq_len.data();
    out->cigar_off = P->cigar_off.data();
    out->n_cigar = P->n_cigar.data();
    out->nm = P->nm.data();
    out->flags = P->flags.data();
    out->n_cigar_ops = P->cigar_ops.size();
    out->cigar_ops = P->cigar_ops.data();
    out->seq_bits = (uint32_t)P->seq_bits;
    out->seq_pool_bytes = P->seq_pool.n;
    out->seq_pool = P->seq_pool.p;
    return PP_OK;
}

extern "C" const char* pp_pack_error(const pp_pack* p) { return p ? p->error.c_str() : "null packer"; }

extern "C" const char* pp_pack_unknown_ref(const pp_pack* p, uint64_t aln) {
    auto it = p->unknown_ref.find(aln);
    return it == p->unknown_ref.end() ? "" : it->second.c_str();
}

extern "C" const char* pp_pack_read_name(const pp_pack* p, uint64_t aln) {
    if (aln >= p->read_id.size()) return "";
    return p->name_pool.c_str() + p->group_name_off[p->read_id[aln]];
}

// The CIGAR of alignment i as text (rebuilt from the packed ops; used only for error messages).
extern "C" int pp_pack_cigar_string(const pp_pack* p, uint64_t aln, char* out, size_t cap) {
    if (!p || !out || cap == 0 || aln >= p->cigar_off.size()) return PP_ERR_ARG;
    std::string s;
    static const char* L = "MIDNSHP=X";
    for (uint32_t i = 0; i < p->n_cigar[aln]; ++i) {
        uint32_t op = p->cigar_ops[p->cigar_off[aln] + i];
        s += std::to_string(op >> 4);
        s += L[(op & 15u) < 9 ? (op & 15u) : 0];
    }
    size_t n = s.size() < cap - 1 ? s.size() : cap - 1;
    memcpy(out, s.data(), n);
    out[n] = 0;
    return PP_OK;
}

extern "C" int pp_pack_file_stats(const pp_pack* p, uint32_t file, uint64_t* alignments, uint64_t* reads) {
    if (!p || file >= p->files.size()) return PP_ERR_ARG;
    if (alignments) *alignments = p->files[file].alignments;
    if (reads) *reads = p->files[file].reads;
    return PP_OK;
}


// ------------------------------------------------------------------------------------------------------
// The 2-bit wire format (pp_abi.h: seq_bits == 2): a read of A/C/G/T only needs 2 bits per base on its way over PCIe; the device
// expands it to the 4-bit codes every kernel works on.  Sequences with any other base (N, IUPAC) stay 4-bit in esc_pool.
// ------------------------------------------------------------------------------------------------------
struct pp_2bit {
    std::vector<uint8_t> flags;
    std::vector<uint32_t> seq_off;
    pp::AlignedBytes pool2, esc;
};

extern "C" int pp_alignments_to_2bit(const pp_alignments* in, pp_alignments* out, pp_2bit** owner) {
    if (!in || !out || !owner || in->seq_bits != 4) return PP_ERR_ARG;
    pp_2bit* W = new pp_2bit();
    const uint64_t n = in->n_aln;
    const uint64_t n_blocks = in->seq_pool_bytes / 16;
    W->flags.assign(in->flags, in->flags + n);
    W->seq_off.assign(in->seq_off, in->seq_off + n);
    W->pool2.resize_zero(n_blocks * 8 + 64);
    std::unordered_map<uint32_t, uint32_t> esc_at;                 // 4-bit block offset of an escaped sequence -> its esc_pool block
    uint64_t esc_blocks = 0;
    // 16 one-hot BAM nibbles (A=1 C=2 G=4 T=8) of one 64-bit word -> 16 two-bit codes (A=0 C=1 G=2 T=3) in 32 bits, word-parallel:
    // code bit 0 = the nibble is C or T (its bits 1 | 3), code bit 1 = G or T (bits 2 | 3); `count` nibbles from the bottom count, the
    // rest (padding past the read's end) must come out as zero.  *ok turns false on a nibble that is not exactly one of the four.
    auto pack16 = [](uint64_t x, uint32_t count, bool* ok) -> uint32_t {
        const uint64_t one = 0x1111111111111111ull;
        const uint64_t keep = count >= 16 ? ~0ull : ((1ull << (4 * count)) - 1ull);
        x &= keep;
        const uint64_t a = x & one, c = (x >> 1) & one, g = (x >> 2) & one, t = (x >> 3) & one;
        if ((a + c + g + t) != (one & keep)) *ok = false;             // per nibble: exactly one bit set (sums stay below 16: no carries)
        uint64_t y = (c | t) | ((g | t) << 1);                         // the code of base i in bits 4i, 4i + 1
        y = (y | (y >> 2)) & 0x0F0F0F0F0F0F0F0Full;
        y = (y | (y >> 4)) & 0x00FF00FF00FF00FFull;
        y = (y | (y >> 8)) & 0x0000FFFF0000FFFFull;
        y = (y | (y >> 16)) & 0x00000000FFFFFFFFull;
        return (uint32_t)y;
    };
    // pass 1, in parallel over ranges of records: every sequence of A/C/G/T only is converted where it stands (a read's blocks are its
    // own); the others are only marked - their order in esc_pool is record order, settled by the sequential pass below
    std::vector<uint8_t> escaped((size_t)n, 0);
    auto convert = [&](uint64_t lo, uint64_t hi) {
        for (uint64_t i = lo; i < hi; ++i) {
            const uint8_t fl = in->flags[i];
            if (fl & (PP_FLAG_SEQSTAR | PP_FLAG_NOSEQ)) continue;   // shares its group's sequence / has none
            const uint32_t off = in->seq_off[i], len = in->seq_len[i];
            const uint8_t* src = in->seq_pool + (size_t)off * 16;
            uint8_t* dst = W->pool2.p + (size_t)off * 8;
            bool plain = true;
            const uint32_t words = (len + 15) / 16;
            for (uint32_t w = 0; w < words; ++w) {
                uint64_t x;
                memcpy(&x, src + 8 * (size_t)w, 8);                 // (little-endian hosts: base j of the word in bits 4j)
                const uint32_t v = pack16(x, std::min<uint32_t>(16, len - 16 * w), &plain);
                memcpy(dst + 4 * (size_t)w, &v, 4);
            }
            if (!plain) {
                escaped[(size_t)i] = 1;
                memset(dst, 0, (size_t)((len + PP_SEQ_BLOCK - 1) / PP_SEQ_BLOCK) * 8);   // nothing reads these blocks; keep them zero
            }
        }
    };
    {
        const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        const unsigned nt = (unsigned)std::min<uint64_t>(std::min(16u, hw), n / 65536 + 1);
        if (nt <= 1) convert(0, n);
        else {
            std::vector<std::thread> th;
            for (unsigned t = 0; t < nt; ++t) th.emplace_back(convert, n * t / nt, n * (t + 1) / nt);
            for (auto& t : th) t.join();
        }
    }
    for (uint64_t i = 0; i < n; ++i) {
        if (!escaped[(size_t)i]) continue;
        const uint32_t off = in->seq_off[i], len = in->seq_len[i];
        const uint64_t blocks = ((uint64_t)len + PP_SEQ_BLOCK - 1) / PP_SEQ_BLOCK;
        W->esc.resize_zero((esc_blocks + blocks) * 16);
        memcpy(W->esc.p + esc_blocks * 16, in->seq_pool + (size_t)off * 16, blocks * 16);
        esc_at.emplace(off, (uint32_t)esc_blocks);
        esc_blocks += blocks;
    }
    if (!esc_at.empty())
        for (uint64_t i = 0; i < n; ++i) {
            if (in->flags[i] & PP_FLAG_NOSEQ) continue;
            auto it = esc_at.find(in->seq_off[i]);
            if (it != esc_at.end()) { W->flags[i] |= PP_FLAG_ESC; W->seq_off[i] = it->second; }
        }
    // Two arrays the device can rebuild stay at home when they are what the packer makes them: CIGAR ops in record order without
    // gaps (cigar_off = prefix sums of n_cigar) and dense group ids (read_id = number of group starts so far - 1).
    bool dense_ops = true, dense_ids = n == 0 || in->read_id[0] == 0;
    {
        uint64_t at = 0;
        for (uint64_t i = 0; i < n && (dense_ops || dense_ids); ++i) {
            if (in->cigar_off[i] != at) dense_ops = false;
            at += in->n_cigar[i];
            if (i && in->read_id[i] != in->read_id[i - 1] && in->read_id[i] != in->read_id[i - 1] + 1) dense_ids = false;
        }
        if (at != in->n_cigar_ops) dense_ops = false;
    }
    if (dense_ids)
        for (uint64_t i = 0; i < n; ++i)
            if (i == 0 || in->read_id[i] != in->read_id[i - 1]) W->flags[i] |= PP_FLAG_NEWGROUP;
    *out = *in;
    if (dense_ops) out->cigar_off = nullptr;
    if (dense_ids) out->read_id = nullptr;
    out->flags = W->flags.data();
    out->seq_off = W->seq_off.data();
    out->seq_bits = 2;
    out->seq_pool = W->pool2.p;
    out->seq_pool_bytes = n_blocks * 8;
    out->esc_pool = W->esc.p;
    out->esc_pool_bytes = esc_blocks * 16;
    *owner = W;
    return PP_OK;
}

extern "C" void pp_2bit_free(pp_2bit* owner) { delete owner; }
