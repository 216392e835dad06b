// filter_pack.cpp — host text side of `polypolish filter`: SAM text -> per-mate record arrays, and the SAM writer.
//
// Restates the TEXT handling of /root/reference/src/filter.rs only:
//   load_alignments_one_file :110-145 with Alignment::new_quick (alignment.rs:102-128): every non-'@' line is parsed
//       (an empty line is "too few columns"), unaligned records are skipped, aligned ones are keyed by QNAME + mate;
//   Alignment::get_ref_end (alignment.rs:138-149) for the read-end coordinate;
//   filter_sam :296-349: headers and unaligned lines verbatim, aligned lines verbatim or with "\tZP:Z:fail" appended,
//       every line terminated by '\n' (CRLF input becomes LF).
// Pairing, thresholds and the pass/fail decision are made on the device (filter_kernels.cu).
#include <cstdio>
#include <string>
#include <string_view>
#include <unordered_map>
#include <vector>

#include "pp_internal.h"

namespace {

struct MateFile {
    std::string path, data;
    std::vector<uint32_t> name_id, contig, ref_start, ref_end;
    std::vector<uint8_t> flags;
    uint64_t n_names_seen = 0;
};

struct Names {
    std::unordered_map<std::string_view, uint32_t> reads, refs;
    uint32_t read_id(std::string_view s) { return reads.emplace(s, (uint32_t)reads.size()).first->second; }
    uint32_t ref_id(std::string_view s) { return refs.emplace(s, (uint32_t)refs.size()).first->second; }
};

// Splits the first 11 tab-separated fields; returns the number found (< 11 means "too few columns").
inline size_t split11(std::string_view s, std::string_view* f) {
    size_t pos = 0, nf = 0;
    while (nf < 11) {
        const char* t = (const char*)memchr(s.data() + pos, '\t', s.size() - pos);
        if (!t) { f[nf++] = s.substr(pos); break; }
        size_t e = (size_t)(t - s.data());
        f[nf++] = s.substr(pos, e - pos);
        pos = e + 1;
    }
    return nf;
}

bool load_mate(MateFile& m, Names& names, std::string& err) {
    if (!pp::read_file(m.path, m.data)) { err = "unable to load alignments from \"" + m.path + "\""; return false; }
    uint64_t line_count = 0;
    bool ok = true;
    std::unordered_map<uint32_t, bool> seen;
    pp::for_each_line(m.data.data(), m.data.size(), [&](std::string_view s) {
        line_count++;
        if (!s.empty() && s[0] == '@') return true;
        std::string_view f[11];
        auto where = [&]() { return " in \"" + m.path + "\" (line " + std::to_string(line_count) + ")"; };
        if (split11(s, f) < 11) { err = "too few columns" + where(); return ok = false; }
        uint64_t flag, pos;
        if (!pp::parse_uint(f[1], 0xFFFFFFFFull, flag)) { err = "invalid FLAG field \"" + std::string(f[1]) + "\"" + where(); return ok = false; }
        if (!pp::parse_uint(f[3], ~0ull, pos)) { err = "invalid POS field \"" + std::string(f[3]) + "\"" + where(); return ok = false; }
        if (flag & 4) return true;                                   // filter.rs:132
        uint64_t start = pos > 0 ? pos - 1 : 0, end;
        if (!pp::cigar_ref_end(f[5], start, end) || end > 0xFFFFFFFEull) { err = "alignment coordinates beyond 2^32 are not supported" + where(); return ok = false; }
        m.name_id.push_back(names.read_id(f[0]));
        m.contig.push_back(names.ref_id(f[2]));
        m.ref_start.push_back((uint32_t)start);
        m.ref_end.push_back((uint32_t)end);
        m.flags.push_back((flag & 16) ? 1 : 0);
        return true;
    });
    return ok;
}

// filter_sam (filter.rs:296-349)
bool write_filtered(const MateFile& m, const uint8_t* pass, const std::string& out_path, uint64_t& n_pass, uint64_t& n_fail) {
    FILE* f = fopen(out_path.c_str(), "wb");
    if (!f) return false;
    std::string buf;
    buf.reserve(1 << 22);
    size_t k = 0;
    n_pass = n_fail = 0;
    bool ok = true;
    pp::for_each_line(m.data.data(), m.data.size(), [&](std::string_view s) {
        bool aligned = false;
        if (!(!s.empty() && s[0] == '@')) {
            const char* t1 = (const char*)memchr(s.data(), '\t', s.size());
            if (t1) {
                size_t b = (size_t)(t1 - s.data()) + 1;
                const char* t2 = (const char*)memchr(s.data() + b, '\t', s.size() - b);
                size_t e = t2 ? (size_t)(t2 - s.data()) : s.size();
                uint64_t flag = 4;
                pp::parse_uint(s.substr(b, e - b), 0xFFFFFFFFull, flag);
                aligned = (flag & 4) == 0;
            }
        }
        buf.append(s.data(), s.size());
        if (aligned) {
            if (pass[k++]) n_pass++;
            else { buf += "\tZP:Z:fail"; n_fail++; }
        }
        buf += '\n';
        if (buf.size() > (1u << 22)) { ok = fwrite(buf.data(), 1, buf.size(), f) == buf.size(); buf.clear(); }
        return ok;
    });
    if (ok && !buf.empty()) ok = fwrite(buf.data(), 1, buf.size(), f) == buf.size();
    return (fclose(f) == 0) && ok;
}

}  // namespace

int pp::check_filter_args(pp_ctx* ctx, const char* in1, const char* in2, const char* out1, const char* out2, const char* orientation,
                          double low, double high, pp_filter_params* prm) {
    {   // check_inputs filter.rs:40-53
        std::vector<std::string> a = {in1, in2};
        if (out1) a.push_back(out1);
        if (out2) a.push_back(out2);
        for (size_t i = 0; i < a.size(); ++i)
            for (size_t j = 0; j < i; ++j)
                if (a[i] == a[j]) return pp_ctx_fail(ctx, PP_ERR_INPUT, "--in1, --in2, --out1 and --out2 must all have unique values");
    }
    if (!(low > 0.0 && low < 50.0)) return pp_ctx_fail(ctx, PP_ERR_INPUT, "--low must be greater than 0 and less than 50");
    if (!(high > 50.0 && high < 100.0)) return pp_ctx_fail(ctx, PP_ERR_INPUT, "--high must be greater than 50 and less than 100");
    const std::string o = orientation;
    prm->orientation = o == "auto" ? -1 : o == "fr" ? 0 : o == "rf" ? 1 : o == "ff" ? 2 : o == "rr" ? 3 : 4;
    prm->low_pct = low;
    prm->high_pct = high;
    prm->n_names = 0;
    return PP_OK;
}

extern "C" int pp_filter_files(pp_ctx* ctx, const char* in1, const char* in2, const char* out1, const char* out2,
                               const char* orientation, double low, double high, int verbose) {
    if (!ctx) return PP_ERR_ARG;
    if (!in1 || !in2 || !out1 || !out2 || !orientation) return pp_ctx_fail(ctx, PP_ERR_ARG, "pp_filter_files: null argument");
    pp_filter_params prm;
    const int arc = pp::check_filter_args(ctx, in1, in2, out1, out2, orientation, low, high, &prm);
    if (arc != PP_OK) return arc;

    pp_filter_result res;
    memset(&res, 0, sizeof res);
    const char* ins[2] = {in1, in2};
    const char* outs[2] = {out1, out2};
    const char* nm[4] = {"fr", "rf", "ff", "rr"};
    auto log_thresholds = [&]() {
        for (int i = 0; i < 4; ++i) fprintf(stderr, "%s: %s pairs\n", nm[i], pp::thousands(res.pairs[i]).c_str());
        fprintf(stderr, "\n%s correct orientation: %s\n\n", prm.orientation < 0 ? "Automatically determined" : "User-specified",
                res.orientation < 4 ? nm[res.orientation] : orientation);
        fprintf(stderr, "Low threshold:  %u\nHigh threshold: %u\n\n", res.low, res.high);
    };

    // Fast path: the SAM text never leaves the device between parse and write (tok_kernels.cu).  PP_TOK_HOST = something the
    // device path leaves to the host code below (malformed line, empty file, ...), which words the reference's messages.
    if (pp_get_parser(ctx) == 0) {
        pp_filter_file_stats fs;
        int rc = pp_filter_files_device(ctx, in1, in2, out1, out2, &prm, &res, &fs, nullptr);
        if (rc == PP_OK) {
            if (verbose) {
                for (int k = 0; k < 2; ++k) fprintf(stderr, "%s: %s alignments\n", ins[k], pp::thousands(fs.alignments[k]).c_str());
                log_thresholds();
                for (int k = 0; k < 2; ++k)
                    fprintf(stderr, "Filtering %s:\n  %s pass\n  %s fail\n\n", ins[k], pp::thousands(fs.pass[k]).c_str(), pp::thousands(fs.fail[k]).c_str());
                fprintf(stderr, "Alignments before filtering: %s\nAlignments after filtering:  %s\n\n", pp::thousands(fs.alignments[0] + fs.alignments[1]).c_str(),
                        pp::thousands(fs.pass[0] + fs.pass[1]).c_str());
                fprintf(stderr, "device text path: %.3f ms (SAM to HBM %.3f ms, filtered SAM to files %.3f ms), %u kernels; filter kernels %.3f ms\n", fs.total_ms,
                        fs.h2d_ms, fs.d2h_ms, fs.launches, res.timing.total_ms);
                fprintf(stderr, "  phases (wall ms): upload+index+parse %.1f, intern+verify+emit %.1f, filter %.1f, output offsets %.1f, output bytes %.1f, download+write %.1f\n",
                        fs.phase_ms[0], fs.phase_ms[1], fs.phase_ms[2], fs.phase_ms[3], fs.phase_ms[4], fs.phase_ms[5]);
            }
            return PP_OK;
        }
        if (rc != PP_TOK_HOST) return rc;
        memset(&res, 0, sizeof res);
    }

    MateFile m[2];
    m[0].path = in1;
    m[1].path = in2;
    Names names;
    std::string err;
    for (int k = 0; k < 2; ++k) {
        if (!load_mate(m[k], names, err)) return pp_ctx_fail(ctx, PP_ERR_INPUT, err.c_str());
        if (verbose) fprintf(stderr, "%s: %s alignments\n", m[k].path.c_str(), pp::thousands(m[k].name_id.size()).c_str());
        if (m[0].name_id.empty() && (k == 0 || m[1].name_id.empty()))      // alignments.is_empty() filter.rs:141-143
            return pp_ctx_fail(ctx, PP_ERR_INPUT, ("no alignments found in \"" + m[k].path + "\"").c_str());
    }

    pp_filter_mate fm[2];
    for (int k = 0; k < 2; ++k) {
        fm[k].n = m[k].name_id.size();
        fm[k].name_id = m[k].name_id.data(); fm[k].contig = m[k].contig.data(); fm[k].ref_start = m[k].ref_start.data();
        fm[k].ref_end = m[k].ref_end.data(); fm[k].flags = m[k].flags.data();
    }
    prm.n_names = names.reads.size();
    std::vector<uint8_t> pass1(fm[0].n + 1), pass2(fm[1].n + 1);
    res.pass1 = pass1.data();
    res.pass2 = pass2.data();
    int rc = pp_filter(ctx, &fm[0], &fm[1], &prm, &res);
    if (rc != PP_OK) return rc;
    if (verbose) log_thresholds();
    uint64_t before = fm[0].n + fm[1].n, after = 0;
    const uint8_t* passes[2] = {pass1.data(), pass2.data()};
    for (int k = 0; k < 2; ++k) {
        uint64_t np, nf;
        if (!write_filtered(m[k], passes[k], outs[k], np, nf))
            return pp_ctx_fail(ctx, PP_ERR_IO, ("unable to write alignments to \"" + std::string(outs[k]) + "\"").c_str());
        after += np;
        if (verbose) fprintf(stderr, "Filtering %s:\n  %s pass\n  %s fail\n\n", m[k].path.c_str(), pp::thousands(np).c_str(), pp::thousands(nf).c_str());
    }
    if (verbose) {
        fprintf(stderr, "Alignments before filtering: %s\nAlignments after filtering:  %s\n\n", pp::thousands(before).c_str(), pp::thousands(after).c_str());
        fprintf(stderr, "device path: %.3f ms, %u kernels\n", res.timing.total_ms, res.timing.launches);
    }
    return PP_OK;
}
