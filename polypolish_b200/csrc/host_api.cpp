// host_api.cpp — whole-command drivers above the C-ABI compute calls.
//
// Mirrors the reference's command drivers (same option checks, same error text, same stdout bytes):
//   polish::polish            /root/reference/src/polish.rs:26-38   (+ :93-134 loading, :137-203 output)
//   filter::filter            /root/reference/src/filter.rs:26-37   (+ :273-349 SAM re-streaming)
// Text (FASTA/SAM) is handled here on the host; all per-alignment / per-position work is behind
// pp_polish() / pp_filter() on the device.  There is no CPU fallback for that work.
#include <chrono>
#include <cmath>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <memory>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "pp_internal.h"

std::string pp::thousands(uint64_t v) {      // num_format Locale::en
    std::string s = std::to_string(v), o;
    int n = (int)s.size();
    for (int i = 0; i < n; ++i) {
        o += s[i];
        if ((n - 1 - i) % 3 == 0 && i != n - 1) o += ',';
    }
    return o;
}

namespace {

// polish.rs:290-300 qscore: "Q∞" at 100 %, "Q0" at or below 0 %, else Q{-10 log10(1 - identity/100)} with two decimals
std::string qscore_text(double identity) {
    if (identity >= 100.0) return "Q\xe2\x88\x9e";
    if (identity <= 0.0) return "Q0";
    const double errors = 1.0 - (identity / 100.0);
    char tmp[64];
    snprintf(tmp, sizeof tmp, "Q%.2f", -10.0 * std::log10(errors));
    return tmp;
}

}  // namespace

extern "C" void pp_free(void* p) { free(p); }

// misc.rs:170-182 complement_base (upper-case input)
static char complement_char(char b) {
    switch (b) {
        case 'A': return 'T'; case 'T': return 'A'; case 'G': return 'C'; case 'C': return 'G'; case 'N': return 'N';
        case 'R': return 'Y'; case 'Y': return 'R'; case 'S': return 'S'; case 'W': return 'W'; case 'K': return 'M'; case 'M': return 'K';
        case 'B': return 'V'; case 'V': return 'B'; case 'D': return 'H'; case 'H': return 'D';
        case '.': return '.'; case '-': return '-'; case '?': return '?';
        default: return 'N';
    }
}

// The string of one "other" allele node (pileup.rs:62 key).
static std::string node_allele(const pp_debug_node& nd, const pp_alignments* a) {
    static const char* NIB = "=ACMGRSVTWYHKDBN";
    std::string out;
    if (a->seq_bits == 4 && (nd.sig & 15)) {
        for (uint32_t i = 0; i < (nd.sig & 15); ++i) out += NIB[(nd.sig >> (4 * (i + 1))) & 15];
        return out;
    }
    if (a->seq_bits == 8 && (nd.sig & 255)) {
        for (uint32_t i = 0; i < (nd.sig & 255); ++i) out += (char)((nd.sig >> (8 * (i + 1))) & 255);
        return out;
    }
    const uint32_t aln = (uint32_t)(nd.val >> 32), start = (uint32_t)(nd.val >> 16) & 0xFFFFu, len = (uint32_t)nd.val & 0xFFFFu;
    const bool rc = a->flags[aln] & PP_FLAG_RC;
    const uint32_t n = a->seq_len[aln];
    for (uint32_t i = 0; i < len; ++i) {
        const uint32_t e = start + i, j = rc ? (n - 1 - e) : e;
        char ch;
        if (a->seq_bits == 4) {
            const uint8_t b = a->seq_pool[(size_t)a->seq_off[aln] * (PP_SEQ_BLOCK / 2) + (j >> 1)];
            ch = NIB[(b >> ((j & 1) * 4)) & 15];
        } else {
            ch = (char)a->seq_pool[(size_t)a->seq_off[aln] * PP_SEQ_BLOCK + j];
        }
        out += rc ? complement_char(ch) : ch;
    }
    return out;
}

// write_debug_header / write_debug_line (polish.rs:247-266) + get_debug_line / get_count_str (pileup.rs:137-166)
static int write_debug_tsv(pp_ctx* ctx, const pp_fasta* fa, const pp_contigs* contigs, const pp_alignments* alns, FILE* f) {
    static const char* STATUS[6] = {"low_depth", "none", "multiple", "too_close", "kept", "changed"};
    const uint64_t G = contigs->off[contigs->n_contigs];
    std::vector<uint32_t> head(G);
    uint64_t n_nodes = 0;
    pp_polish_debug_alleles(ctx, nullptr, nullptr, 0, &n_nodes);           // size query (reports the node count, then fails on the null buffers)
    std::vector<pp_debug_node> nodes(n_nodes + 1);
    int rc = pp_polish_debug_alleles(ctx, head.data(), nodes.data(), n_nodes, &n_nodes);
    if (rc != PP_OK) return rc;
    if (fputs("name\tpos\tbase\tdepth\tinvalid\tvalid\tpileup\tstatus\tnew_base\n", f) < 0) return PP_ERR_IO;
    const uint64_t CH = 1 << 18;
    std::vector<pp_debug_pos> recs(CH);
    std::string buf;
    std::vector<std::string> counts;
    char tmp[64];
    for (uint32_t c = 0; c < contigs->n_contigs; ++c) {
        const char* name = pp_fasta_name(fa, c);
        for (uint64_t p0 = contigs->off[c]; p0 < contigs->off[c + 1]; p0 += CH) {
            const uint64_t n = std::min<uint64_t>(CH, contigs->off[c + 1] - p0);
            rc = pp_polish_debug_fetch(ctx, p0, n, recs.data());
            if (rc != PP_OK) return rc;
            buf.clear();
            for (uint64_t i = 0; i < n; ++i) {
                const pp_debug_pos& r = recs[i];
                const uint64_t gp = p0 + i;
                counts.clear();
                static const char* ACGT = "ACGT";
                for (int b = 0; b < 4; ++b) if (r.count[b]) counts.push_back(std::string(1, ACGT[b]) + "x" + std::to_string(r.count[b]));
                if (r.count[4]) counts.push_back("-x" + std::to_string(r.count[4]));
                if (r.count[5]) counts.push_back(std::string(1, (char)r.original) + "x" + std::to_string(r.count[5]));
                for (uint32_t nd = head[gp]; nd != 0;) {
                    const pp_debug_node& node = nodes[nd - 1];
                    counts.push_back(node_allele(node, alns) + "x" + std::to_string(node.count));
                    nd = node.next == 0xFFFFFFFFu ? 0 : node.next + 1;
                }
                std::sort(counts.begin(), counts.end());
                buf += name; buf += '\t'; buf += std::to_string(gp - contigs->off[c]); buf += '\t'; buf += (char)r.original; buf += '\t';
                snprintf(tmp, sizeof tmp, "%.1f", r.depth);          // Rust {:.1}: both round the exact binary value
                buf += tmp; buf += '\t'; buf += std::to_string(r.invalid_threshold); buf += '\t'; buf += std::to_string(r.valid_threshold); buf += '\t';
                for (size_t k = 0; k < counts.size(); ++k) { if (k) buf += ','; buf += counts[k]; }
                buf += '\t'; buf += STATUS[r.status < 6 ? r.status : 0]; buf += '\t';
                if (r.new_node != 0xFFFFFFFFu) buf += node_allele(nodes[r.new_node], alns); else buf += (char)r.new_char;
                buf += '\n';
            }
            if (fwrite(buf.data(), 1, buf.size(), f) != buf.size()) return PP_ERR_IO;
        }
    }
    return PP_OK;
}

// One shard on one GPU (run by its own host thread when there are several).
struct ShardJob {
    pp_ctx* ctx = nullptr;
    pp_contigs contigs;
    pp_alignments alns;
    const uint32_t* contig_map = nullptr;
    bool resident = false;               // the dataset is already on the device (device tokeniser)
    std::vector<uint64_t> out_off, changed, zero;
    std::vector<double> tdepth;
    std::vector<uint8_t> bases;
    pp_polish_result res;
    int rc = PP_OK;
    std::string err;
    // a shard made on the device (every GPU tokenises the text itself): the shard's contigs live here
    std::vector<uint32_t> own_map, own_local;
    std::vector<uint64_t> own_off;
    std::vector<uint8_t> own_bases;
};

static void run_shard(ShardJob* j, const pp_polish_params* prm) {
    const uint64_t G = j->contigs.off[j->contigs.n_contigs];
    j->out_off.assign(j->contigs.n_contigs + 1, 0);
    j->changed.assign(j->contigs.n_contigs, 0);
    j->zero.assign(j->contigs.n_contigs, 0);
    j->tdepth.assign(j->contigs.n_contigs, 0.0);
    memset(&j->res, 0, sizeof j->res);
    // Output is at most G + inserted bases; start with G + 1 MiB and retry once with the exact size.
    uint64_t cap = G + (1u << 20);
    for (int attempt = 0; attempt < 2; ++attempt) {
        j->bases.resize(cap);
        j->res.out_off = j->out_off.data();
        j->res.out_bases = j->bases.data();
        j->res.out_cap = cap;
        j->res.changed = j->changed.data();
        j->res.zero_depth = j->zero.data();
        j->res.total_depth = j->tdepth.data();
        j->rc = j->resident ? pp_polish_resident(j->ctx, prm, &j->res) : pp_polish(j->ctx, &j->contigs, &j->alns, prm, &j->res);
        if (j->rc == PP_ERR_ARG && j->res.out_len > cap) { cap = j->res.out_len; continue; }
        break;
    }
    if (j->rc != PP_OK) j->err = pp_last_error(j->ctx);
}

// Every job, one host thread per GPU.  true: one of them met a data error (PP_ERR_INPUT), whose message needs read / reference names,
// which only the host packer has.
static bool run_jobs(std::vector<ShardJob>& jobs, const pp_polish_params* prm) {
    std::vector<std::thread> th;
    for (size_t s = 1; s < jobs.size(); ++s) th.emplace_back(run_shard, &jobs[s], prm);
    run_shard(&jobs[0], prm);
    for (auto& t : th) t.join();
    for (const ShardJob& j : jobs)
        if (j.rc == PP_ERR_INPUT) return true;
    return false;
}

// The resident dataset of a context copied back into host arrays (pp_dataset_download), for the allele strings of the --debug TSV.
// Plain new[] without value initialisation: the copy overwrites every byte, so zero-filling 0.4 GB first would only cost time.
struct HostCopy {
    std::unique_ptr<uint32_t[]> contig, ref_start, read_id, seq_off, cigar_off, nm, cigar_ops;
    std::unique_ptr<uint16_t[]> seq_len, n_cigar;
    std::unique_ptr<uint8_t[]> flags, seq_pool;
    int fetch(pp_ctx* ctx, pp_alignments* v) {
        int rc = pp_dataset_sizes(ctx, v);
        if (rc != PP_OK) return rc;
        const size_t n = (size_t)v->n_aln + 1;
        contig.reset(new uint32_t[n]); ref_start.reset(new uint32_t[n]); read_id.reset(new uint32_t[n]); seq_off.reset(new uint32_t[n]);
        cigar_off.reset(new uint32_t[n]); nm.reset(new uint32_t[n]); seq_len.reset(new uint16_t[n]); n_cigar.reset(new uint16_t[n]);
        flags.reset(new uint8_t[n]); cigar_ops.reset(new uint32_t[(size_t)v->n_cigar_ops + 1]); seq_pool.reset(new uint8_t[(size_t)v->seq_pool_bytes + 64]);
        v->contig = contig.get(); v->ref_start = ref_start.get(); v->read_id = read_id.get(); v->seq_off = seq_off.get();
        v->cigar_off = cigar_off.get(); v->nm = nm.get(); v->seq_len = seq_len.get(); v->n_cigar = n_cigar.get(); v->flags = flags.get();
        v->cigar_ops = cigar_ops.get(); v->seq_pool = seq_pool.get();
        return pp_dataset_download(ctx, v);
    }
};

// Cuts a SAM file into n byte ranges for n GPUs: cut[0] = 0, cut[n] = size, every other cut is the start of a line whose QNAME differs from
// the line before it (a read group - consecutive lines of one QNAME, alignment.rs:214-272 - is never split).  false: not a plain file,
// or a line longer than the window (the caller lets one GPU read the whole file instead).
static bool split_ranges(const char* path, int n, std::vector<uint64_t>& cut) {
    const int fd = open(path, O_RDONLY);
    if (fd < 0) return false;
    struct stat sb;
    if (fstat(fd, &sb) != 0 || !S_ISREG(sb.st_mode)) { close(fd); return false; }
    const uint64_t S = (uint64_t)sb.st_size;
    cut.assign((size_t)n + 1, S);
    cut[0] = 0;
    const size_t W = 1 << 20;
    std::vector<char> buf(W);
    bool ok = true;
    // the line starting at `pos` (a line start): its QNAME and where the next line starts
    auto line_at = [&](uint64_t pos, std::string& qname, uint64_t& next) -> bool {
        if (pos >= S) return false;
        const size_t want = (size_t)std::min<uint64_t>(W, S - pos);
        size_t got = 0;
        while (got < want) {
            const ssize_t r = pread(fd, buf.data() + got, want - got, (off_t)(pos + got));
            if (r <= 0) { ok = false; return false; }
            got += (size_t)r;
        }
        const char* nl = (const char*)memchr(buf.data(), '\n', got);
        if (!nl && pos + got < S) { ok = false; return false; }                  // longer than the window
        const size_t len = nl ? (size_t)(nl - buf.data()) : got;
        const char* tab = (const char*)memchr(buf.data(), '\t', len);
        qname.assign(buf.data(), tab ? (size_t)(tab - buf.data()) : len);
        next = pos + len + 1;
        return true;
    };
    for (int g = 1; g < n && ok; ++g) {
        uint64_t pos = std::max<uint64_t>(S / (uint64_t)n * (uint64_t)g, cut[g - 1]);
        if (pos >= S) { cut[g] = S; continue; }
        // the first line start at or after pos
        if (pos > 0) {
            std::string q; uint64_t nx = 0;
            if (!line_at(pos - 1, q, nx)) { if (!ok) break; cut[g] = S; continue; }       // (the rest of the line that holds byte pos - 1)
            pos = std::min(nx, S);
        }
        // ... then on to the first line whose QNAME differs from its predecessor's
        std::string qa, qb;
        uint64_t na = 0, nb = 0;
        if (!line_at(pos, qa, na)) { if (!ok) break; cut[g] = S; continue; }
        uint64_t cand = std::min(na, S);
        for (;;) {
            if (cand >= S || !line_at(cand, qb, nb)) { cand = S; break; }
            if (qb != qa || (!qb.empty() && qb[0] == '@')) break;
            qa.swap(qb);
            cand = std::min(nb, S);
        }
        if (!ok) break;
        cut[g] = std::max(cand, cut[g - 1]);
    }
    close(fd);
    return ok;
}

extern "C" int pp_sam_split_ranges(const char* path, int n, uint64_t* cuts) {
    if (!path || n < 1 || !cuts) return PP_ERR_ARG;
    if (pp::is_bam(path)) return PP_ERR_IO;                          // byte ranges of a BAM are not record boundaries
    std::vector<uint64_t> c;
    if (!split_ranges(path, n, c)) return PP_ERR_IO;
    std::copy(c.begin(), c.end(), cuts);
    return PP_OK;
}

template <auto Free> struct Freer { template <class T> void operator()(T* p) const { Free(p); } };
using FastaPtr = std::unique_ptr<pp_fasta, Freer<pp_fasta_free>>;
using PackPtr = std::unique_ptr<pp_pack, Freer<pp_pack_free>>;
using ShardsPtr = std::unique_ptr<pp_shards, Freer<pp_shards_free>>;

// What a loader hands the driver: one job per shard; the alignments as the host sees them (the count always, the arrays where the
// host holds them: the packer's, or the --debug download); the per-file log, printed only once the load has succeeded, and the
// timing lines; and the owners of what the jobs point into.
struct Loaded {
    std::vector<ShardJob> jobs;
    pp_alignments alns{};
    std::string log, timing;
    PackPtr pk;
    ShardsPtr shards;
    HostCopy copy;
    void one_job(pp_ctx* ctx, const pp_contigs& contigs, bool resident) {       // the whole assembly on one GPU
        jobs.assign(1, ShardJob());
        jobs[0].ctx = ctx; jobs[0].contigs = contigs; jobs[0].alns = alns; jobs[0].resident = resident;
    }
};

// A device tokenisation with 4-bit bases, once more with 8-bit bases when the text needs them (PP_TOK_NEED8); past that the host decides.
template <class F> static int with_seq_bits(F&& tokenise) {
    int rc = tokenise(4);
    if (rc == PP_TOK_NEED8) rc = tokenise(8);
    return rc == PP_TOK_NEED8 ? PP_TOK_HOST : rc;
}

// `filter` in front of `polish` in the same call (pp_filter_polish_files): the two SAM files are `sams`, this says what to filter with
struct FusedFilter {
    pp_filter_params prm;
    const char* orientation;
    const char *out1, *out2;             // filtered SAM files, or null: not written
};

// filter (filter.rs:26-37) and the load of polish in one pass over the text: both files go to HBM once, the filter's verdict
// becomes the ZP flag of the tokenised records (what ZP:Z:fail does after a round trip through two files).
static int load_fused(pp_ctx* ctx, const pp_fasta* fa, const pp_contigs& contigs, const char* const* sams, const FusedFilter& ff,
                      int careful, Loaded& d) {
    pp_filter_result fres{};
    pp_filter_file_stats fs;
    pp_fused_polish fuse{};
    fuse.fasta = fa; fuse.careful = careful;
    int rc = pp_filter_files_device(ctx, sams[0], sams[1], ff.out1, ff.out2, &ff.prm, &fres, &fs, &fuse);
    if (rc == PP_OK && fuse.rc == PP_TOK_HOST) rc = PP_TOK_HOST;
    if (rc != PP_OK) return rc;
    static const char* nm[4] = {"fr", "rf", "ff", "rr"};
    char tmp[512];
    for (int k = 0; k < 2; ++k) {
        snprintf(tmp, sizeof tmp, "%s: %s alignments, %s pass the insert-size filter, %s fail\n", sams[k], pp::thousands(fs.alignments[k]).c_str(),
                 pp::thousands(fs.pass[k]).c_str(), pp::thousands(fs.fail[k]).c_str());
        d.log += tmp;
    }
    snprintf(tmp, sizeof tmp, "orientation %s, insert size thresholds %u - %u\n", fres.orientation < 4 ? nm[fres.orientation] : ff.orientation, fres.low, fres.high);
    d.log += tmp;
    d.alns.n_aln = fuse.n_aln;
    d.one_job(ctx, contigs, true);
    return PP_OK;
}

// Several GPUs, no host in the middle: the host only decides which contig goes where (longest contig first onto the lightest shard)
// and where to cut the files; the text, the records and the shards never pass through host memory as arrays.  Every GPU reads ITS
// byte range of every file (cut between read groups), tokenises it, and the read groups are exchanged between the GPUs
// (tok_kernels.cu pp_tok_exchange_finish): 1/N of the text per PCIe link.  A BAM file is inflated once, here, and every GPU decodes
// its range of the records of that one image (cut between read groups as well).
static int load_device_ranges(pp_ctx* const* ctxs, uint32_t n_shards, const pp_fasta* fa, const pp_contigs& contigs,
                              const char* const* sams, int n_sams, int careful, Loaded& d) {
    std::vector<uint32_t> order(contigs.n_contigs), owner(contigs.n_contigs);
    for (uint32_t i = 0; i < contigs.n_contigs; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return contigs.off[x + 1] - contigs.off[x] > contigs.off[y + 1] - contigs.off[y]; });
    std::vector<uint64_t> load(n_shards, 0);
    for (uint32_t ci : order) {
        const uint32_t best = (uint32_t)(std::min_element(load.begin(), load.end()) - load.begin());
        owner[ci] = best;
        load[best] += contigs.off[ci + 1] - contigs.off[ci];
    }
    d.jobs.assign(n_shards, ShardJob());
    for (uint32_t s = 0; s < n_shards; ++s) {
        ShardJob& j = d.jobs[s];
        j.ctx = ctxs[s];
        j.own_local.assign(contigs.n_contigs, 0xFFFFFFFFu);
        j.own_off.assign(1, 0);
        for (uint32_t ci = 0; ci < contigs.n_contigs; ++ci) {
            if (owner[ci] != s) continue;
            j.own_local[ci] = (uint32_t)j.own_map.size();
            j.own_map.push_back(ci);
            j.own_bases.insert(j.own_bases.end(), contigs.bases + contigs.off[ci], contigs.bases + contigs.off[ci + 1]);
            j.own_off.push_back(j.own_bases.size());
        }
        j.contigs.n_contigs = (uint32_t)j.own_map.size(); j.contigs.off = j.own_off.data(); j.contigs.bases = j.own_bases.data();
        j.contig_map = j.own_map.data();
        j.resident = true;
    }
    std::vector<std::vector<uint64_t>> cuts((size_t)n_sams);
    std::vector<std::unique_ptr<pp::BamImage>> bams((size_t)n_sams);
    for (int i = 0; i < n_sams; ++i) {
        if (pp::is_bam(sams[i])) {
            bams[(size_t)i].reset(new pp::BamImage());
            std::string err;
            if (pp::bam_load(sams[i], fa, *bams[(size_t)i], err) != PP_OK) return PP_TOK_HOST;     // the host path words the error
            pp::bam_split(*bams[(size_t)i], (int)n_shards, cuts[(size_t)i]);
        } else if (!split_ranges(sams[i], (int)n_shards, cuts[(size_t)i])) {
            return PP_TOK_HOST;
        }
    }
    std::vector<std::vector<pp_tok_stats>> tst(n_shards, std::vector<pp_tok_stats>((size_t)n_sams));
    int rc = with_seq_bits([&](int bits) {
        std::vector<int> trc(n_shards, PP_OK);
        auto work = [&](uint32_t s) {
            pp_ctx* c = ctxs[s];
            std::vector<uint64_t> off((size_t)n_sams), len((size_t)n_sams);
            uint64_t mine = 0;
            for (int i = 0; i < n_sams; ++i) {
                if (bams[(size_t)i]) continue;                          // (a BAM's range is a range of records, set below)
                off[(size_t)i] = cuts[(size_t)i][s]; len[(size_t)i] = cuts[(size_t)i][s + 1] - cuts[(size_t)i][s]; mine += len[(size_t)i];
            }
            int r = pp_tok_begin(c, fa, careful ? 1 : 0, bits);
            if (r == PP_OK) r = pp_tok_expect(c, mine);
            if (r == PP_OK) r = pp_tok_set_ranges(c, off.data(), len.data(), n_sams);
            for (int i = 0; i < n_sams && r == PP_OK; ++i)
                if (bams[(size_t)i]) r = pp_tok_set_bam_range(c, i, bams[(size_t)i].get(), cuts[(size_t)i][s], cuts[(size_t)i][s + 1]);
            if (r == PP_OK) r = pp_tok_add_files(c, sams, n_sams, tst[s].data());
            trc[s] = r;
            if (r != PP_OK && r != PP_TOK_HOST && r != PP_TOK_NEED8) d.jobs[s].err = pp_last_error(c);
        };
        std::vector<std::thread> tt;
        for (uint32_t s = 1; s < n_shards; ++s) tt.emplace_back(work, s);
        work(0);
        for (auto& t : tt) t.join();
        for (int want : {PP_TOK_HOST, PP_TOK_NEED8})
            for (uint32_t s = 0; s < n_shards; ++s) if (trc[s] == want) return want;
        for (uint32_t s = 0; s < n_shards; ++s)
            if (trc[s] != PP_OK) return pp_ctx_fail(ctxs[0], trc[s], d.jobs[s].err.c_str());
        return PP_OK;
    });
    if (rc != PP_OK) return rc;
    bool empty_file = false;
    for (int i = 0; i < n_sams; ++i) {
        uint64_t na = 0, nr = 0, nl = 0;
        float h2d = 0, dev = 0;
        for (uint32_t s = 0; s < n_shards; ++s) {
            const pp_tok_stats& t = tst[s][(size_t)i];
            na += t.alignments; nr += t.reads; nl += t.lines; h2d = std::max(h2d, t.h2d_ms); dev = std::max(dev, t.device_ms);
        }
        empty_file |= na == 0;                                         // "no alignments in <file>" (alignment.rs:268-270): the host path words it
        d.log += std::string(sams[i]) + ": " + pp::thousands(na) + " alignments from " + pp::thousands(nr) + " reads\n";
        char tmp[256];
        if (bams[(size_t)i])
            snprintf(tmp, sizeof tmp, "BAM decoder %s: %s records in %u ranges, read %.3f ms, inflate %.3f ms, record walk %.3f ms, image to HBM %.3f ms, "
                     "kernels %.3f ms (slowest GPU)\n", sams[i], pp::thousands(nl).c_str(), n_shards, bams[(size_t)i]->read_ms, bams[(size_t)i]->inflate_ms,
                     bams[(size_t)i]->walk_ms, h2d, dev);
        else
            snprintf(tmp, sizeof tmp, "SAM tokeniser %s: %s lines in %u byte ranges, text to HBM %.3f ms, kernels %.3f ms (slowest GPU)\n", sams[i],
                     pp::thousands(nl).c_str(), n_shards, h2d, dev);
        d.timing += tmp;
    }
    if (empty_file) return PP_TOK_HOST;
    std::vector<const uint32_t*> lo(n_shards);
    std::vector<pp_contigs> sc(n_shards);
    for (uint32_t s = 0; s < n_shards; ++s) { lo[s] = d.jobs[s].own_local.data(); sc[s] = d.jobs[s].contigs; }
    const auto t0 = std::chrono::steady_clock::now();
    rc = pp_tok_exchange_finish(ctxs, (int)n_shards, owner.data(), contigs.n_contigs, lo.data(), sc.data(), &d.alns.n_aln);
    if (rc != PP_OK) return rc;
    char tmp[160];
    snprintf(tmp, sizeof tmp, "read groups exchanged between %u GPUs and binned: %.3f ms\n", n_shards,
             std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count());
    d.timing += tmp;
    for (uint32_t s = 0; s < n_shards; ++s) {
        pp_alignments v;
        if (pp_dataset_sizes(ctxs[s], &v) == PP_OK) d.jobs[s].alns.n_aln = v.n_aln;
    }
    return PP_OK;
}

// SAM files -> resident dataset of one context through the device tokeniser (tok_kernels.cu).  `log` collects the per-file lines
// add_to_pileup prints (alignment.rs:266-271).  With --debug the dataset is also copied back: the TSV's allele strings are read there.
static int load_device_one(pp_ctx* ctx, const pp_fasta* fa, const pp_contigs& contigs, const char* const* sams, int n_sams, int careful,
                           bool debug, Loaded& d) {
    uint64_t total = 0;
    for (int i = 0; i < n_sams; ++i) total += pp::file_size(sams[i]);
    std::vector<pp_tok_stats> st((size_t)n_sams);
    int rc = with_seq_bits([&](int bits) {
        int r = pp_tok_begin(ctx, fa, careful ? 1 : 0, bits);
        if (r == PP_OK) r = pp_tok_expect(ctx, total);
        if (r == PP_OK) r = pp_tok_add_files(ctx, sams, n_sams, st.data());
        return r;
    });
    if (rc == PP_OK) rc = pp_tok_finish(ctx);
    if (rc == PP_OK && debug) rc = d.copy.fetch(ctx, &d.alns);
    if (rc != PP_OK) return rc;
    d.alns.n_aln = 0;
    for (int i = 0; i < n_sams; ++i) {
        d.alns.n_aln += st[i].alignments;
        d.log += std::string(sams[i]) + ": " + pp::thousands(st[i].alignments) + " alignments from " + pp::thousands(st[i].reads) + " reads\n";
        char tmp[320];
        float rd = 0, inf = 0, walk = 0, up = 0;
        if (pp_tok_bam_phases(ctx, i, &rd, &inf, &walk, &up))
            snprintf(tmp, sizeof tmp, "BAM decoder %s: %s records, read %.3f ms, inflate %.3f ms, record walk %.3f ms, image to HBM %.3f ms, %u kernels %.3f ms\n",
                     sams[i], pp::thousands(st[i].lines).c_str(), rd, inf, walk, up, st[i].launches, st[i].device_ms);
        else
            snprintf(tmp, sizeof tmp, "SAM tokeniser %s: %s lines, text to HBM %.3f ms, %u kernels %.3f ms\n", sams[i], pp::thousands(st[i].lines).c_str(),
                     st[i].h2d_ms, st[i].launches, st[i].device_ms);
        d.timing += tmp;
    }
    d.one_job(ctx, contigs, true);
    return PP_OK;
}

// The host packer (sam_pack.cpp), which words every error of the text the way the reference does, then the host sharder (shard.cpp)
// when there are several shards.  Each file's line is printed as soon as the file is parsed, as add_to_pileup does (alignment.rs:266-271).
static int load_host(pp_ctx* const* ctxs, uint32_t n_shards, const pp_fasta* fa, const pp_contigs& contigs, const char* const* sams, int n_sams,
                     int careful, int verbose, Loaded& d) {
    d.pk.reset(pp_pack_create(fa, careful));
    int rc = PP_OK;
    for (int i = 0; i < n_sams && rc == PP_OK; ++i) {
        rc = pp_pack_add_sam_file(d.pk.get(), sams[i]);
        if (rc == PP_OK && verbose) {
            uint64_t na = 0, nr = 0;
            pp_pack_file_stats(d.pk.get(), (uint32_t)i, &na, &nr);
            fprintf(stderr, "%s: %s alignments from %s reads\n", sams[i], pp::thousands(na).c_str(), pp::thousands(nr).c_str());
        }
    }
    if (rc == PP_OK) rc = pp_pack_finish(d.pk.get(), &d.alns);
    if (rc != PP_OK) return pp_ctx_fail(ctxs[0], rc, pp_pack_error(d.pk.get()));
    if (n_shards == 1) { d.one_job(ctxs[0], contigs, false); return PP_OK; }
    d.jobs.assign(n_shards, ShardJob());
    d.shards.reset(pp_shards_build(&contigs, &d.alns, n_shards));
    for (uint32_t s = 0; s < n_shards; ++s) {
        d.jobs[s].ctx = ctxs[s];
        pp_shards_get(d.shards.get(), s, &d.jobs[s].contigs, &d.jobs[s].alns, &d.jobs[s].contig_map, nullptr);
    }
    return PP_OK;
}

// The message of a failed job; a device-detected data error is re-worded with the names the reference prints
// (alignment.rs:190-198,298-300), which `pk` can look up when the job ran over its unsharded arrays.
static std::string job_error(const ShardJob& j, pp_pack* pk) {
    std::string m = j.err;
    if (!pk || j.rc != PP_ERR_INPUT || j.res.error_aln < 0) return m;
    const char* rn = pp_pack_read_name(pk, (uint64_t)j.res.error_aln);
    if (m.rfind("query name", 0) == 0)
        return "query name " + std::string(pp_pack_unknown_ref(pk, (uint64_t)j.res.error_aln)) + " in SAM but not in assembly";
    if (m.rfind("CIGAR string does not", 0) == 0)
        return "CIGAR string for read " + std::string(rn) + " does not match read sequence";
    if (m.rfind("unexpected character", 0) == 0) {
        char cg[4096];
        pp_pack_cigar_string(pk, (uint64_t)j.res.error_aln, cg, sizeof cg);
        return "unexpected character (other than M, =, X, I or D) in CIGAR string for read " + std::string(rn) +
               ": \"" + cg + "\" - did you use BWA MEM to generate your alignments?";
    }
    return m + " (read " + std::string(rn) + ")";
}

// print_seq_to_stdout polish.rs:196-203, contigs in input order (polish.rs:147-152), with the per-contig report (polish.rs:205-226)
static int emit(pp_ctx* ctx, const pp_fasta* fa, const pp_contigs& contigs, const Loaded& d, int verbose, char** out_fasta, uint64_t* out_len) {
    const std::vector<ShardJob>& jobs = d.jobs;
    // where each input contig's polished bases are: (job, local contig)
    std::vector<std::pair<uint32_t, uint32_t>> where(contigs.n_contigs);
    for (uint32_t s = 0; s < jobs.size(); ++s)
        for (uint32_t lc = 0; lc < jobs[s].contigs.n_contigs; ++lc)
            where[jobs.size() == 1 ? lc : jobs[s].contig_map[lc]] = {s, lc};
    std::string out;
    uint64_t total = 0;
    for (auto& j : jobs) total += j.res.out_len;
    out.reserve(total + 128 * (size_t)contigs.n_contigs);
    for (uint32_t i = 0; i < contigs.n_contigs; ++i) {
        const ShardJob& j = jobs[where[i].first];
        const uint32_t lc = where[i].second;
        out += '>';
        out += pp_fasta_name(fa, i);
        const char* desc = pp_fasta_description(fa, i);
        if (desc[0]) { out += ' '; out += desc; }
        out += " polypolish\n";
        out.append((const char*)j.bases.data() + j.out_off[lc], j.out_off[lc + 1] - j.out_off[lc]);
        out += '\n';
        if (verbose) {
            uint64_t len = contigs.off[i + 1] - contigs.off[i];
            fprintf(stderr, "Polishing %s (%s bp):\n", pp_fasta_name(fa, i), pp::thousands(len).c_str());
            fprintf(stderr, "  mean read depth: %.1fx\n", j.tdepth[lc] / (double)len);                       // polish.rs:208-210
            fprintf(stderr, "  %s bp %s a depth of zero (%.4f%% coverage)\n", pp::thousands(j.zero[lc]).c_str(), j.zero[lc] == 1 ? "has" : "have",
                    100.0 * (double)(len - j.zero[lc]) / (double)len);
            fprintf(stderr, "  %s %s changed (%.4f%% of total positions)\n", pp::thousands(j.changed[lc]).c_str(),
                    j.changed[lc] == 1 ? "position" : "positions", 100.0 * (double)j.changed[lc] / (double)len);
            const double accuracy = 100.0 - 100.0 * (double)j.changed[lc] / (double)len;
            fprintf(stderr, "  estimated pre-polishing sequence accuracy: %.4f%% (%s)\n\n", accuracy, qscore_text(accuracy).c_str());
        }
    }
    if (verbose) {
        fputs(d.timing.c_str(), stderr);
        for (uint32_t s = 0; s < jobs.size(); ++s) {
            const pp_timing& t = jobs[s].res.timing;
            fprintf(stderr, "GPU job %u: %u contigs, %s alignments; device path %.3f ms (h2d + binning %.3f, goodness/k %.3f, tile %.3f, compact %.3f, d2h %.3f), %u kernels\n",
                    s, jobs[s].contigs.n_contigs, pp::thousands(jobs[s].alns.n_aln).c_str(), t.total_ms, t.stage_ms[6], t.stage_ms[2], t.stage_ms[3],
                    t.stage_ms[4], t.stage_ms[7], t.launches);
        }
    }
    char* buf = (char*)malloc(out.size() + 1);
    if (!buf) return pp_ctx_fail(ctx, PP_ERR_NOMEM, "out of memory");
    memcpy(buf, out.data(), out.size());
    buf[out.size()] = 0;
    *out_fasta = buf;
    *out_len = out.size();
    return PP_OK;
}

// polish::polish (polish.rs:26-38) over one or several GPUs (contigs shard across them, SURVEY.md §8e).  With `ff`, filter runs in
// front of it on the device; PP_TOK_HOST then means that the two commands have to run through files instead (pp_filter_polish_files).
static int polish_files_impl(pp_ctx* const* ctxs, int n_ctx, const char* assembly, const char* const* sams, int n_sams,
                             const pp_polish_params* prm, const char* debug_path, char** out_fasta, uint64_t* out_len, int verbose,
                             const FusedFilter* ff = nullptr) {
    pp_ctx* ctx = ctxs[0];
    if (!assembly || !prm || !out_fasta || !out_len || n_sams < 0) return pp_ctx_fail(ctx, PP_ERR_ARG, "pp_polish_files: bad arguments");
    *out_fasta = nullptr;
    *out_len = 0;
    // check_option_values polish.rs:277-287
    if (!(prm->fraction_valid > 0.0 && prm->fraction_valid < 1.0)) return pp_ctx_fail(ctx, PP_ERR_INPUT, "--fraction_valid must be between 0 and 1 (exclusive)");
    if (!(prm->fraction_invalid > 0.0 && prm->fraction_invalid < 1.0)) return pp_ctx_fail(ctx, PP_ERR_INPUT, "--fraction_invalid must be between 0 and 1 (exclusive)");
    if (prm->fraction_invalid >= prm->fraction_valid) return pp_ctx_fail(ctx, PP_ERR_INPUT, "--fraction_invalid must be less than --fraction_valid");
    // check_inputs_exist polish.rs:269-274
    if (!pp::file_exists(assembly)) return pp_ctx_fail(ctx, PP_ERR_INPUT, ("\"" + std::string(assembly) + "\" file does not exist").c_str());
    for (int i = 0; i < n_sams; ++i)
        if (!pp::file_exists(sams[i])) return pp_ctx_fail(ctx, PP_ERR_INPUT, ("\"" + std::string(sams[i]) + "\" file does not exist").c_str());
    const bool debug = debug_path && debug_path[0];
    FILE* debug_file = nullptr;
    if (debug) {                                          // create_debug_file polish.rs:230-244
        debug_file = fopen(debug_path, "wb");
        if (!debug_file) return pp_ctx_fail(ctx, PP_ERR_IO, ("unable to create \"" + std::string(debug_path) + "\"").c_str());
    }
    struct FileCloser { FILE*& f; ~FileCloser() { if (f) fclose(f); } } closer{debug_file};

    const bool device_parser = n_sams > 0 && pp_get_parser(ctx) == 0;
    // the first SAM file starts streaming into HBM while the assembly is loaded
    if (device_parser && n_ctx == 1) pp_tok_prefetch(ctx, sams[0]);
    char ebuf[1024];
    FastaPtr fa(pp_fasta_load(assembly, ebuf, sizeof ebuf));
    if (!fa) return pp_ctx_fail(ctx, PP_ERR_INPUT, ebuf);
    pp_contigs contigs;
    pp_fasta_view(fa.get(), &contigs);
    if (verbose) {
        fprintf(stderr, "Loading assembly\n");
        for (uint32_t i = 0; i < contigs.n_contigs; ++i)
            fprintf(stderr, "%s (%s bp)\n", pp_fasta_name(fa.get(), i), pp::thousands(contigs.off[i + 1] - contigs.off[i]).c_str());
        fprintf(stderr, "\nLoading alignments\n");
    }

    // one job per GPU; with one GPU the job is the whole assembly
    const uint32_t n_shards = debug ? 1u : (uint32_t)std::max(1, std::min<int>(n_ctx, (int)contigs.n_contigs));   // the debug TSV is written from one GPU
    if (debug) pp_polish_set_debug(ctx, 1);
    // The SAM text is parsed in HBM (tok_kernels.cu) first.  Anything unusual - PP_TOK_HOST, or a data error raised by the polish
    // kernels - repeats the load with the host packer, which decides.
    Loaded d;
    int rc = PP_TOK_HOST;
    if (device_parser) {
        if (ff) rc = load_fused(ctx, fa.get(), contigs, sams, *ff, prm->careful, d);
        else if (n_shards > 1) rc = load_device_ranges(ctxs, n_shards, fa.get(), contigs, sams, n_sams, prm->careful, d);
        else rc = load_device_one(ctx, fa.get(), contigs, sams, n_sams, prm->careful, debug, d);
        if (rc == PP_OK && run_jobs(d.jobs, prm)) rc = PP_TOK_HOST;
    }
    if (rc == PP_TOK_HOST) {
        if (ff) return PP_TOK_HOST;
        d = Loaded();
        rc = load_host(ctxs, n_shards, fa.get(), contigs, sams, n_sams, prm->careful, verbose, d);
        if (rc != PP_OK) return rc;
        if (run_jobs(d.jobs, prm) && d.jobs.size() > 1) {
            // the message names the read of the offending line: its index in the unsharded arrays is what the packer can look up,
            // so the job runs once more as one shard
            d.shards.reset();
            d.one_job(ctx, contigs, false);
            run_shard(&d.jobs[0], prm);
        }
    } else if (rc != PP_OK) {
        return rc;
    }
    if (verbose) fputs(d.log.c_str(), stderr);

    uint64_t n_used = 0;
    for (const ShardJob& j : d.jobs) {
        n_used += j.res.n_aln_used;
        if (j.rc != PP_OK) { rc = pp_ctx_fail(ctx, j.rc, job_error(j, d.jobs.size() == 1 ? d.pk.get() : nullptr).c_str()); break; }
    }
    if (debug) pp_polish_set_debug(ctx, rc == PP_OK ? 2 : 0);      // keep the recorded data readable, stop recording
    if (rc == PP_OK && debug) {
        rc = write_debug_tsv(ctx, fa.get(), &contigs, &d.alns, debug_file);
        if (rc != PP_OK && rc != PP_ERR_CUDA) rc = pp_ctx_fail(ctx, PP_ERR_IO, ("unable to write to file \"" + std::string(debug_path) + "\"").c_str());
    }
    if (rc != PP_OK) return rc;
    if (verbose) {
        fprintf(stderr, "\nFiltering for high-quality end-to-end alignments%s:\n", prm->careful ? " from reads with only one alignment" : "");
        fprintf(stderr, "  %s alignments kept\n", pp::thousands(n_used).c_str());
        fprintf(stderr, "  %s alignments discarded\n\n", pp::thousands(d.alns.n_aln - n_used).c_str());
    }
    return emit(ctx, fa.get(), contigs, d, verbose, out_fasta, out_len);
}

// filter::filter (filter.rs:26-37) then polish::polish (polish.rs:26-38) on its output, as one call: same FASTA as running the two
// commands through intermediate files, which are only written when the caller names them.
extern "C" int pp_filter_polish_files(pp_ctx* ctx, const char* assembly, const char* in1, const char* in2, const char* out1, const char* out2,
                                      const char* orientation, double low, double high, const pp_polish_params* prm, char** out_fasta,
                                      uint64_t* out_len, int verbose) {
    if (!ctx) return PP_ERR_ARG;
    if (!in1 || !in2 || !orientation) return pp_ctx_fail(ctx, PP_ERR_ARG, "pp_filter_polish_files: null argument");
    FusedFilter ff;
    int rc = pp::check_filter_args(ctx, in1, in2, out1, out2, orientation, low, high, &ff.prm);
    if (rc != PP_OK) return rc;
    ff.orientation = orientation; ff.out1 = out1; ff.out2 = out2;
    const char* sams[2] = {in1, in2};
    rc = polish_files_impl(&ctx, 1, assembly, sams, 2, prm, nullptr, out_fasta, out_len, verbose, &ff);
    if (rc != PP_TOK_HOST) return rc;
    // Something the fused device path leaves to the text code (a malformed line, an empty file, host parsing asked for, a data
    // error whose message needs names): the two commands one after the other, through files, exactly like the reference.
    std::string t1 = out1 ? out1 : "", t2 = out2 ? out2 : "";
    char tmpl1[] = "/tmp/polypolish_filtered_1_XXXXXX", tmpl2[] = "/tmp/polypolish_filtered_2_XXXXXX";
    if (t1.empty()) { int fd = mkstemp(tmpl1); if (fd < 0) return pp_ctx_fail(ctx, PP_ERR_IO, "unable to create a temporary file for the filtered alignments"); close(fd); t1 = tmpl1; }
    if (t2.empty()) { int fd = mkstemp(tmpl2); if (fd < 0) return pp_ctx_fail(ctx, PP_ERR_IO, "unable to create a temporary file for the filtered alignments"); close(fd); t2 = tmpl2; }
    rc = pp_filter_files(ctx, in1, in2, t1.c_str(), t2.c_str(), orientation, low, high, verbose);
    if (rc == PP_OK) {
        const char* fsams[2] = {t1.c_str(), t2.c_str()};
        rc = polish_files_impl(&ctx, 1, assembly, fsams, 2, prm, nullptr, out_fasta, out_len, verbose);
    }
    if (!out1) unlink(t1.c_str());
    if (!out2) unlink(t2.c_str());
    return rc;
}

extern "C" int pp_polish_files(pp_ctx* ctx, const char* assembly, const char* const* sams, int n_sams,
                               const pp_polish_params* prm, const char* debug_path, char** out_fasta,
                               uint64_t* out_len, int verbose) {
    return pp_polish_files_multi(&ctx, 1, assembly, sams, n_sams, prm, debug_path, out_fasta, out_len, verbose);
}

// Several GPUs of one box: contigs shard across the contexts (one host thread each); errors are reported on ctxs[0].
extern "C" int pp_polish_files_multi(pp_ctx* const* ctxs, int n_ctx, const char* assembly, const char* const* sams, int n_sams,
                                     const pp_polish_params* prm, const char* debug_path, char** out_fasta,
                                     uint64_t* out_len, int verbose) {
    if (!ctxs || n_ctx < 1 || !ctxs[0]) return PP_ERR_ARG;
    return polish_files_impl(ctxs, n_ctx, assembly, sams, n_sams, prm, debug_path, out_fasta, out_len, verbose);
}
