// bam_rec.h — per-record logic of the BAM decoder (SAMv1 §4.2), host + device.
//
// A BAM record is decoded into the same tok::LineRec the SAM tokeniser's parse_line (tok_line.h) makes of the record's SAM
// line, so that the scans, the group heads and the group close of tok_kernels.cu run unchanged.  The record's SAM line is
// what bam.cpp renders (QNAME .. QUAL, NM and ZP tags, CG folded into the CIGAR); the host packer parses that line and stays
// the authority: whatever needs wording (a bad CIGAR op, a negative NM, the long-CIGAR placeholder, a structural fault) is
// answered with LK_HOST here.  tests/bam_harness.cpp runs these bodies on the CPU against the host packer.
#pragma once
#include "tok_line.h"

namespace tok {

constexpr uint32_t BAM_FIXED = 36;            // block_size through tlen
enum : uint8_t { BF_OK = 0, BF_PAST_BLOCK = 1, BF_REF_RANGE = 2, BF_AUX = 3 };

// little-endian loads at any byte offset (records are not 4-byte aligned)
TK_HD uint32_t le16(Txt& x, uint64_t p) { return (uint32_t)x.at(p) | ((uint32_t)x.at(p + 1) << 8); }
TK_HD uint32_t le32(Txt& x, uint64_t p) { return le16(x, p) | (le16(x, p + 2) << 16); }

struct BamFix {
    uint32_t block_size, l_name, mapq, bin, n_cigar, flag, l_seq;
    int32_t ref, pos, next_ref, next_pos, tlen;
};

TK_HD void bam_fixed(Txt& x, uint64_t s, BamFix& f) {
    f.block_size = le32(x, s);
    f.ref = (int32_t)le32(x, s + 4);
    f.pos = (int32_t)le32(x, s + 8);
    f.l_name = x.at(s + 12);
    f.mapq = x.at(s + 13);
    f.bin = le16(x, s + 14);
    f.n_cigar = le16(x, s + 16);
    f.flag = le16(x, s + 18);
    f.l_seq = le32(x, s + 20);
    f.next_ref = (int32_t)le32(x, s + 24);
    f.next_pos = (int32_t)le32(x, s + 28);
    f.tlen = (int32_t)le32(x, s + 32);
}

// Offset of the aux data from the record start (64-bit: l_seq is a u32 of the file).
TK_HD uint64_t bam_aux_rel(const BamFix& f) {
    return BAM_FIXED + f.l_name + 4ull * f.n_cigar + ((uint64_t)f.l_seq + 1) / 2 + (uint64_t)f.l_seq;
}

// Bytes of one aux value of a fixed-size type, 0 for the others.
TK_HD uint32_t aux_size(uint8_t t) {
    switch (t) {
        case 'A': case 'c': case 'C': return 1;
        case 's': case 'S': return 2;
        case 'i': case 'I': case 'f': return 4;
        default: return 0;
    }
}

TK_HD int64_t aux_int(Txt& x, uint64_t p, uint8_t t) {
    switch (t) {
        case 'c': return (int8_t)x.at(p);
        case 'C': return x.at(p);
        case 's': return (int16_t)le16(x, p);
        case 'S': return le16(x, p);
        case 'i': return (int32_t)le32(x, p);
        default: return le32(x, p);   // 'I'
    }
}

TK_HD bool is_int_type(uint8_t t) { return t == 'c' || t == 'C' || t == 's' || t == 'S' || t == 'i' || t == 'I'; }

// What polish reads of the aux data: NM of an integer type (NM:i:<decimal> in SAM; the last one wins), ZP:Z:fail in any case,
// and the CG:B:I array of a long CIGAR.
struct BamAux {
    uint32_t nm;          // 0xFFFFFFFF: none (the text path's own "missing" value, which NM:i:4294967295 also gives)
    bool nm_neg;          // an NM below zero: "invalid NM tag" in the text path
    bool zp_fail;
    bool zp_odd;          // a ZP:Z value with a tab, CR or LF, which would change how its SAM line splits
    bool cg;
    uint64_t cg_pos;      // first element of CG:B:I
    uint32_t cg_n;
};

// Walks the aux fields [p, e).  false: a field runs past e, or a type that SAMv1 does not define.
TK_HD bool bam_aux(Txt& x, uint64_t p, uint64_t e, BamAux& a) {
    a.nm = 0xFFFFFFFFu; a.nm_neg = false; a.zp_fail = false; a.zp_odd = false; a.cg = false; a.cg_pos = 0; a.cg_n = 0;
    while (p < e) {
        if (e - p < 3) return false;
        const uint8_t t0 = x.at(p), t1 = x.at(p + 1), ty = x.at(p + 2);
        p += 3;
        const uint32_t fs = aux_size(ty);
        if (fs) {
            if (e - p < fs) return false;
            if (t0 == 'N' && t1 == 'M' && is_int_type(ty)) {
                const int64_t v = aux_int(x, p, ty);
                if (v < 0) a.nm_neg = true;
                else a.nm = (uint32_t)v;
            }
            p += fs;
        } else if (ty == 'Z' || ty == 'H') {
            const bool zp = ty == 'Z' && lower(t0) == 'z' && lower(t1) == 'p';
            uint64_t q = p;
            bool odd = false;
            while (q < e) {
                const uint8_t c = x.at(q);
                if (c == 0) break;
                odd |= c == '\t' || c == '\n' || c == '\r';
                ++q;
            }
            if (q >= e) return false;                                       // no NUL before the end of the record
            if (zp) {
                a.zp_odd |= odd;
                if (q - p == 4 && lower(x.at(p)) == 'f' && lower(x.at(p + 1)) == 'a' && lower(x.at(p + 2)) == 'i' && lower(x.at(p + 3)) == 'l')
                    a.zp_fail = true;
            }
            p = q + 1;
        } else if (ty == 'B') {
            if (e - p < 5) return false;
            const uint8_t sub = x.at(p);
            const uint64_t n = le32(x, p + 1), es = aux_size(sub);
            if (es == 0 || sub == 'A' || (e - p - 5) / es < n) return false;
            if (t0 == 'C' && t1 == 'G' && sub == 'I') { a.cg = true; a.cg_pos = p + 5; a.cg_n = (uint32_t)n; }
            p += 5 + n * es;
        } else {
            return false;
        }
    }
    return true;
}

// The structural checks of one record at s, inside a stream of n bytes (the record walk has checked that 4 + block_size bytes
// are there).  BF_OK or the fault; a is filled when BF_OK.
TK_HD uint8_t bam_check(Txt& x, uint64_t s, const BamFix& f, uint32_t n_ref, BamAux& a) {
    const uint64_t rel = bam_aux_rel(f);
    if (f.block_size < BAM_FIXED - 4 || rel > 4ull + f.block_size) return BF_PAST_BLOCK;
    if (f.ref < -1 || f.ref >= (int64_t)n_ref || f.next_ref < -1 || f.next_ref >= (int64_t)n_ref) return BF_REF_RANGE;
    if (!bam_aux(x, s + rel, s + 4 + f.block_size, a)) return BF_AUX;
    return BF_OK;
}

// Is the CIGAR the long-CIGAR placeholder kSmN (SAMv1 §4.2.2)?
TK_HD bool bam_placeholder(Txt& x, uint64_t s, const BamFix& f) {
    if (f.n_cigar != 2) return false;
    const uint64_t c = s + BAM_FIXED + f.l_name;
    return le32(x, c) == ((f.l_seq << 4) | PP_OP_S) && (le32(x, c + 4) & 15u) == PP_OP_N;
}

// One record at s -> LineRec, as parse_line would make it of the record's SAM line.  ref_contig[ref + 1] = contig of refID ref
// (entry 0 is refID -1, RNAME "*").  fault: the structural fault behind an LK_HOST, else BF_OK.
TK_HD uint8_t parse_bam(Txt& x, uint64_t s, const uint32_t* ref_contig, uint32_t n_ref, LineRec& r, uint8_t& fault) {
    r.contig = PP_CONTIG_UNKNOWN; r.ref_start = 0; r.nm = 0; r.nops = 0; r.slen = 0; r.cig_rel = 0; r.seq_rel = 0;
    r.name_len = 0; r.cig_len = 0; r.flags = 0; r.kind = LK_SKIP; r.need8 = 0; r.pad = 0;
    BamFix f;
    bam_fixed(x, s, f);
    BamAux a;
    fault = bam_check(x, s, f, n_ref, a);
    if (fault != BF_OK) return LK_HOST;
    const bool aligned = (f.flag & 4) == 0;
    // QNAME: a name that starts with '@' makes a header line of the record, a tab or LF splits it differently
    const uint32_t nl = f.l_name ? f.l_name - 1 : 0;
    for (uint32_t k = 0; k < nl; ++k) {
        const uint8_t c = x.at(s + BAM_FIXED + k);
        if (c == '\t' || c == '\n' || (k == 0 && c == '@')) return LK_HOST;
    }
    if (f.pos < -1) return LK_HOST;                                         // "invalid POS field"
    if (bam_placeholder(x, s, f)) return LK_HOST;
    const uint64_t c0 = s + BAM_FIXED + f.l_name;
    uint32_t nops = 0;
    for (uint32_t k = 0; k < f.n_cigar; ++k) {
        const uint32_t op = le32(x, c0 + 4ull * k);
        if ((op & 15u) > PP_OP_X) return LK_HOST;                           // "invalid CIGAR string"
        if (op >> 4) nops++;
    }
    if (a.nm_neg) return LK_HOST;                                           // "invalid NM tag"
    if (a.zp_odd) return LK_HOST;
    if (a.nm == 0xFFFFFFFFu && aligned) return LK_HOST;                     // "missing NM tag"
    if (!aligned) return LK_SKIP;                                           // alignment.rs:250
    if (nops == 0 || f.l_seq > 0xFFFFu) return LK_HOST;
    r.contig = ref_contig[f.ref + 1];
    r.ref_start = f.pos > 0 ? (uint32_t)f.pos : 0u;                         // POS = pos + 1; POS 0 stays 0 (alignment.rs:58-61)
    r.nm = a.nm;
    r.nops = nops;
    r.slen = f.l_seq;
    r.cig_rel = BAM_FIXED + f.l_name;
    r.cig_len = f.n_cigar;
    r.seq_rel = BAM_FIXED + f.l_name + 4 * f.n_cigar;
    r.name_len = nl;
    const bool star = f.l_seq == 0;
    r.flags = (uint8_t)(((f.flag & 16) ? PP_FLAG_REVERSE : 0) | (a.zp_fail ? PP_FLAG_ZPFAIL : 0) | (star ? PP_FLAG_SEQSTAR : 0));
    r.kind = LK_ALIGNED;
    return LK_ALIGNED;
}

// Second visit of an aligned record: its CIGAR words as stored, zero-length operations dropped.
TK_HD void emit_bam_cigar(Txt& x, uint64_t s, const LineRec& r, uint32_t* ops) {
    uint32_t k = 0;
    for (uint32_t i = 0; i < r.cig_len && k < r.nops; ++i) {
        const uint32_t op = le32(x, s + r.cig_rel + 4ull * i);
        if (op >> 4) ops[k++] = op;
    }
}

// ... and its bases: BAM keeps base 2k in the high nibble, the pool in the low one, so each byte has its nibbles swapped (4-bit
// pool), or becomes the letters of "=ACMGRSVTWYHKDBN" (8-bit pool).  Code 0 ('=') has no 4-bit pool code: returns true then.
template <int BITS>
TK_HD bool emit_bam_seq(Txt& x, uint64_t s, const LineRec& r, uint8_t* dst) {
    const uint64_t b = s + r.seq_rel;
    const uint32_t n = r.slen, nblk = seq_blocks(r), nbytes = (n + 1) / 2;
    bool exotic = false;
    for (uint32_t blk = 0; blk < nblk; ++blk) {
        if (BITS == 4) {
            uint64_t w[2] = {0, 0};
            for (uint32_t k = 0; k < 16; ++k) {
                const uint32_t q = blk * 16 + k;
                if (q >= nbytes) break;
                const uint8_t c = x.at(b + q);
                const uint8_t hi = c >> 4, lo = c & 15;
                exotic |= hi == 0 || (2 * q + 1 < n && lo == 0);
                const uint8_t sw = (uint8_t)(hi | (2 * q + 1 < n ? (uint8_t)(lo << 4) : 0));
                w[k >> 3] |= (uint64_t)sw << (8 * (k & 7));
            }
            uint64_t* d = reinterpret_cast<uint64_t*>(dst + (size_t)blk * 16);
            d[0] = w[0]; d[1] = w[1];
        } else {
            const char* L = "=ACMGRSVTWYHKDBN";
            for (uint32_t wi = 0; wi < 4; ++wi) {
                uint64_t v = 0;
                for (uint32_t j = 0; j < 8; ++j) {
                    const uint32_t q = blk * 32 + wi * 8 + j;
                    if (q < n) {
                        const uint8_t c = x.at(b + (q >> 1));
                        v |= (uint64_t)(uint8_t)L[(q & 1) ? (c & 15) : (c >> 4)] << (8 * j);
                    }
                }
                reinterpret_cast<uint64_t*>(dst + (size_t)blk * 32)[wi] = v;
            }
        }
    }
    return exotic;
}

}  // namespace tok
