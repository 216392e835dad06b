// pp_internal.h — shared host-side declarations of libpolypolish_b200 (not part of the ABI).
#pragma once
#include <cstdint>
#include <cstring>
#include <string>
#include <string_view>
#include <unordered_map>
#include <vector>

#include "../../include/pp_abi.h"

namespace pp {

// Rust str::lines() over a byte buffer without allocating: split on '\n', strip one '\r' before it;
// a final unterminated line is a line (alignment.rs:238, misc.rs:109).
template <class F>
inline void for_each_line(const char* data, size_t n, F&& f) {
    size_t pos = 0;
    while (pos < n) {
        const char* nl = (const char*)memchr(data + pos, '\n', n - pos);
        size_t end = nl ? (size_t)(nl - data) : n;
        size_t e2 = end;
        if (nl && e2 > pos && data[e2 - 1] == '\r') e2--;
        if (!f(std::string_view(data + pos, e2 - pos))) return;
        if (!nl) break;
        pos = end + 1;
    }
}

bool read_file(const std::string& path, std::string& out);
bool read_gz_file(const std::string& path, std::string& out);
bool file_exists(const std::string& path);
uint64_t file_size(const std::string& path);   // 0 when it cannot be stat'ed

// Rust "123".parse::<u32/usize>(): optional '+', >= 1 ASCII digit, overflow is an error.
bool parse_uint(std::string_view s, uint64_t maxv, uint64_t& out);

// Alignment::get_ref_end (alignment.rs:138-149): tolerant scan of \d+[MIDNSHP=X] tokens.
bool cigar_ref_end(std::string_view cigar, uint64_t start, uint64_t& end);

// 16-byte aligned growable byte buffer (sequence pool).
struct AlignedBytes {
    uint8_t* p = nullptr;
    size_t n = 0, cap = 0;
    ~AlignedBytes();
    void reserve(size_t want);
    void resize_zero(size_t want);  // grow to `want`, new bytes zeroed
    void clear() { n = 0; }
};

// 1234567 -> "1,234,567" (num_format Locale::en, what the reference's logs print)
std::string thousands(uint64_t v);

// The argument checks of `polypolish filter` (check_inputs filter.rs:40-53, the --low / --high ranges) and its parameters, the
// orientation text as a code.  out1 / out2 may be null (not written).  PP_OK, or the error, reported on ctx.
int check_filter_args(pp_ctx* ctx, const char* in1, const char* in2, const char* out1, const char* out2, const char* orientation,
                      double low, double high, pp_filter_params* prm);

}  // namespace pp

struct pp_fasta {
    std::vector<std::string> names, descriptions;
    std::vector<uint64_t> off;     // n+1
    std::string bases;             // upper-cased, concatenated
    std::unordered_map<std::string, uint32_t> index;
};

struct pp_pack {
    const pp_fasta* fasta = nullptr;
    bool careful = false;
    int seq_bits = 4;
    bool need8 = false;
    std::string error;
    int error_code = 0;

    // SoA (pp_alignments)
    std::vector<uint32_t> contig, ref_start, read_id, seq_off, cigar_off, nm;
    std::vector<uint16_t> seq_len, n_cigar;
    std::vector<uint8_t> flags;
    std::vector<uint32_t> cigar_ops;
    pp::AlignedBytes seq_pool;
    uint64_t seq_blocks = 0;       // pool length in PP_SEQ_BLOCK units

    // names for error messages
    std::string name_pool;                 // QNAMEs, NUL separated
    std::vector<uint64_t> group_name_off;  // [n_reads]
    std::unordered_map<uint64_t, std::string> unknown_ref;

    struct FileStat { std::string name; uint64_t alignments = 0, reads = 0; };
    std::vector<FileStat> files;

    // sources kept so that an 8-bit repack can re-run them
    struct Source { bool is_file; std::string path_or_name; std::string text; };
    std::vector<Source> sources;
    bool replaying = false;
    bool no_replay = false;
    unsigned threads = 0;          // parsing threads for files (0 = hardware)
    size_t min_chunk = 8u << 20;   // smallest chunk of a file one parsing thread gets
    void* stream = nullptr;        // open streaming file (sam_pack.cpp)
    std::string tmp;
};

int pp_ctx_fail(pp_ctx* ctx, int code, const char* msg);

// `polypolish filter` with the SAM text handled on the device (tok_kernels.cu); what the log of pp_filter_files prints.
struct pp_filter_file_stats {
    uint64_t alignments[2], pass[2], fail[2], text_bytes[2], out_bytes[2];
    float h2d_ms, d2h_ms, total_ms;
    float phase_ms[6];     // wall: 0 upload+index+parse, 1 intern+verify+emit, 2 filter proper, 3 output lengths+scan, 4 output bytes, 5 download+write
    uint32_t launches;
};
// filter + polish without the intermediate files: the request to tokenise the resident texts for polish, and what came of it
struct pp_fused_polish {
    const pp_fasta* fasta;
    int careful;
    pp_tok_stats stats[2];
    uint64_t n_aln;
    int rc;                // PP_OK: the filtered alignments are the resident dataset; PP_TOK_HOST: the host text path must do it
};
int pp_filter_files_device(pp_ctx* ctx, const char* in1, const char* in2, const char* out1, const char* out2, const pp_filter_params* prm,
                           pp_filter_result* res, pp_filter_file_stats* fs, pp_fused_polish* fuse);
