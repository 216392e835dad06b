// CPU harness for the device BAM decoder's per-record logic (polypolish_b200/csrc/bam_rec.h): runs k_bam_parse's and
// k_bam_emit's bodies record by record, then the shared group passes of tok_line.h, in the order of the device pipeline, so
// that tests/test_bam_cpu.py can compare the arrays with the host packer's without a GPU.  Compiled by the test with g++.
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "../polypolish_b200/csrc/bam_rec.h"

// stream: the inflated BAM (magic onward), n bytes.  ref_contig: [n_ref + 1] as pp::BamImage holds it.  Returns PP_OK,
// PP_TOK_HOST (counts[5] = first record the device leaves to the host) or PP_TOK_NEED8; counts[0..3] = aln, ops, blk, reads.
extern "C" int bam_cpu(const uint8_t* stream, uint64_t n, const uint32_t* ref_contig, uint32_t n_ref, int careful, int bits,
                       uint64_t cap_aln, uint64_t cap_ops, uint64_t cap_seq_bytes, uint32_t* contig, uint32_t* ref_start,
                       uint32_t* read_id, uint32_t* seq_off, uint16_t* seq_len, uint32_t* cigar_off, uint16_t* n_cigar, uint32_t* nm,
                       uint8_t* flags, uint32_t* cigar_ops, uint8_t* seq_pool, uint64_t* counts) {
    std::vector<uint64_t> buf(n / 8 + 16, 0);                  // 8-byte aligned, zero padded (what the device text buffer is)
    uint8_t* d = reinterpret_cast<uint8_t*>(buf.data());
    memcpy(d, stream, n);
    tok::Txt x(d);
    // header, then the block_size chain
    uint64_t p = 8 + tok::le32(x, 4);
    const uint32_t nr = tok::le32(x, p);
    p += 4;
    for (uint32_t r = 0; r < nr; ++r) p += 4 + tok::le32(x, p) + 4;
    std::vector<uint64_t> rec;
    while (p + 4 <= n) { rec.push_back(p); p += 4 + tok::le32(x, p); }
    const uint64_t R = rec.size();
    counts[4] = R;
    counts[5] = ~0ull;
    std::vector<tok::LineRec> recs(R);
    std::vector<uint64_t> s_al(R + 1, 0), s_ops(R + 1, 0), s_blk(R + 1, 0);
    for (uint64_t i = 0; i < R; ++i) {
        uint8_t fault;
        const uint8_t kind = tok::parse_bam(x, rec[i], ref_contig, n_ref, recs[i], fault);
        const bool al = kind == tok::LK_ALIGNED;
        s_al[i] = al; s_ops[i] = al ? recs[i].nops : 0; s_blk[i] = al ? tok::seq_blocks(recs[i]) : 0;
        if (kind == tok::LK_HOST && counts[5] == ~0ull) counts[5] = i;
    }
    if (counts[5] != ~0ull) return PP_TOK_HOST;
    auto exscan = [](std::vector<uint64_t>& v) { uint64_t run = 0; for (auto& e : v) { uint64_t t = e; e = run; run += t; } };
    exscan(s_al); exscan(s_ops); exscan(s_blk);
    const uint64_t n_al = s_al[R], n_ops = s_ops[R], n_blk = s_blk[R];
    if (n_al == 0) return PP_TOK_HOST;
    const uint64_t A0 = counts[0], O0 = counts[1], B0 = counts[2], R0 = counts[3];
    const uint64_t blk_bytes = bits == 4 ? 16 : 32;
    if (A0 + n_al > cap_aln || O0 + n_ops > cap_ops || (B0 + n_blk) * blk_bytes > cap_seq_bytes) return PP_ERR_ARG;
    std::vector<uint64_t> name_pos(n_al);
    std::vector<uint32_t> name_len(n_al), head(n_al);
    bool need8 = false;
    for (uint64_t i = 0; i < R; ++i) {
        const tok::LineRec& r = recs[i];
        if (r.kind != tok::LK_ALIGNED) continue;
        const uint64_t s = rec[i], la = s_al[i], A = A0 + la, co = O0 + s_ops[i], bo = B0 + s_blk[i];
        const bool star = r.flags & PP_FLAG_SEQSTAR;
        contig[A] = r.contig; ref_start[A] = r.ref_start; seq_off[A] = star ? 0u : (uint32_t)bo; seq_len[A] = (uint16_t)r.slen;
        cigar_off[A] = (uint32_t)co; n_cigar[A] = (uint16_t)r.nops; nm[A] = r.nm; flags[A] = r.flags;
        name_pos[la] = s + tok::BAM_FIXED; name_len[la] = r.name_len;
        tok::emit_bam_cigar(x, s, r, cigar_ops + co);
        if (bits == 4) { if (tok::emit_bam_seq<4>(x, s, r, seq_pool + bo * 16)) need8 = true; }
        else tok::emit_bam_seq<8>(x, s, r, seq_pool + bo * 32);
    }
    for (uint64_t a = 0; a < n_al; ++a) head[a] = tok::group_head(x, a, 0, name_pos.data(), name_len.data()) ? 1u : 0u;
    uint32_t run = 0;
    bool group_err = false;
    for (uint64_t a = 0; a < n_al; ++a) {
        run += head[a];
        read_id[A0 + a] = (uint32_t)(R0 + run - 1);
    }
    for (uint64_t a = 0; a < n_al; ++a)
        if (head[a] && !tok::close_group(a, n_al, head.data(), careful != 0, seq_off + A0, seq_len + A0, flags + A0)) group_err = true;
    if (group_err) return PP_TOK_HOST;
    if (need8 && bits == 4) return PP_TOK_NEED8;
    counts[0] = A0 + n_al; counts[1] = O0 + n_ops; counts[2] = B0 + n_blk; counts[3] = R0 + run;
    return PP_OK;
}
