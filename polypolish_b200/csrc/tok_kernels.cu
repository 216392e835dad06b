// tok_kernels.cu — SAM text -> packed alignments ON THE DEVICE (SURVEY.md §8f-1, "GPU SAM tokeniser / packer").
//
// The text of one SAM file is streamed into HBM (pinned double buffers, several reader threads) and turned into exactly the
// arrays the host packer (sam_pack.cpp) would have produced, so that `polypolish polish` spends its time on PCIe instead
// of on a host parse:
//
//   k_tok_count   newlines per 16 KiB tile                                   text read once      (HBM-bound)
//   (cub scan)    tile offsets
//   k_tok_index   line starts                                                text read once
//   k_tok_parse   one thread per line: columns, FLAG/POS/NM/ZP, CIGAR check, RNAME -> contig     text read once
//   (cub scans)   alignment index, CIGAR-pool offset, sequence-pool offset of every line
//   k_tok_emit    one thread per aligned line: record arrays, CIGAR ops, 4-bit (or 8-bit) bases   CIGAR+SEQ read again
//   k_tok_heads   one thread per alignment: does it open a read group (QNAME compare with its predecessor)
//   (cub scan)    read ids
//   k_tok_groups  one thread per group head: SEQ="*" records take the group's source sequence
//
// A BAM file (bam.cpp: inflated on the host into one image with its record offsets) takes a second front end: the image goes up
// through the same pinned slots, k_bam_parse (one thread per record, bam_rec.h) stands in for the three line passes and
// k_bam_emit for k_tok_emit; the scans, k_tok_heads and k_tok_groups are shared.
//
// Per-item logic lives in tok_line.h (host+device, CPU-tested against the host packer).  The host packer stays the
// authority on everything unusual: a malformed line, a limit, a group without sequence make the call return PP_TOK_HOST and
// the caller runs pp_pack_* on the same text, which yields the result or the reference's own error message
// (alignment.rs:49-98, 225-346).
#include <cuda_runtime.h>

#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/statvfs.h>
#include <unistd.h>

#include <cerrno>
#include <algorithm>
#include <atomic>
#include <chrono>
#include <string>
#include <thread>
#include <vector>

#include "pp_ctx.cuh"
#include "tok_line.h"
#include "tok_table.h"
#include "tok_strip.h"
#include "bam_rec.h"

// A temporary that does not fit in device memory is not an error of the data: the host text code takes over.
#define TRY_ALLOC(x) do { if ((x) != cudaSuccess) { cudaGetLastError(); return PP_TOK_HOST; } } while (0)

namespace {

constexpr int TK_TILE = 16384;        // bytes of text per CTA in the newline passes
constexpr int TK_THREADS = 256;
constexpr int TK_LINE_THREADS = 128;  // threads (= lines) per CTA in the per-line passes
constexpr int TK_READERS = 16;        // at most this many host threads stream a file into the device
constexpr size_t TK_SLOT = 4u << 20;  // pinned bytes per slot (two slots per reader)
constexpr size_t TK_LOOK = 1u << 20;  // QUAL-stripping upload: how far past its nominal slice a reader looks for the line end

struct TokStatus {
    unsigned long long first_bad;     // smallest line index the device does not accept (~0 = none)
    unsigned int need8;               // a SEQ byte outside the 4-bit alphabet
    unsigned int group_err;           // a read group without any sequence (alignment.rs:319-321)
};

struct TokTable {                     // device pointers of the contig-name table and the nibble table
    tok::ContigTable ct;
    const uint8_t* nibtab;
};

__device__ __forceinline__ uint32_t newline_mask(uint32_t w) { return __vcmpeq4(w, 0x0A0A0A0Au); }

__global__ void __launch_bounds__(TK_THREADS) k_tok_count(const uint8_t* __restrict__ text, uint64_t n16, unsigned long long* __restrict__ tile_cnt) {
    const uint64_t t0 = (uint64_t)blockIdx.x * TK_TILE;
    uint32_t c = 0;
    for (uint32_t off = threadIdx.x * 16; off < TK_TILE; off += TK_THREADS * 16) {
        const uint64_t p = t0 + off;
        if (p < n16) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(text + p));
            c += __popc(newline_mask(v.x) & 0x01010101u) + __popc(newline_mask(v.y) & 0x01010101u) +
                 __popc(newline_mask(v.z) & 0x01010101u) + __popc(newline_mask(v.w) & 0x01010101u);
        }
    }
    typedef cub::BlockReduce<uint32_t, TK_THREADS> BR;
    __shared__ typename BR::TempStorage tmp;
    const uint32_t s = BR(tmp).Sum(c);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = s;
}

// line_start[i] = offset of the first byte of line i; line_start[0] = 0, line_start[k+1] = position after newline k.
__global__ void __launch_bounds__(TK_THREADS) k_tok_index(const uint8_t* __restrict__ text, uint64_t n16, const unsigned long long* __restrict__ tile_off,
                                                          unsigned long long* __restrict__ line_start) {
    typedef cub::BlockScan<uint32_t, TK_THREADS> BS;
    __shared__ typename BS::TempStorage tmp;
    const uint64_t t0 = (uint64_t)blockIdx.x * TK_TILE;
    unsigned long long run = tile_off[blockIdx.x];
    if (blockIdx.x == 0 && threadIdx.x == 0) line_start[0] = 0;
    for (uint32_t it = 0; it < TK_TILE / (TK_THREADS * 16); ++it) {
        const uint64_t p = t0 + (uint64_t)it * TK_THREADS * 16 + threadIdx.x * 16;
        uint32_t m[4] = {0, 0, 0, 0};
        if (p < n16) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(text + p));
            m[0] = newline_mask(v.x) & 0x01010101u; m[1] = newline_mask(v.y) & 0x01010101u;
            m[2] = newline_mask(v.z) & 0x01010101u; m[3] = newline_mask(v.w) & 0x01010101u;
        }
        const uint32_t cnt = __popc(m[0]) + __popc(m[1]) + __popc(m[2]) + __popc(m[3]);
        uint32_t ex, total;
        BS(tmp).ExclusiveSum(cnt, ex, total);
        __syncthreads();
        unsigned long long o = run + ex;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t mk = m[k];
            while (mk) {
                const uint32_t b = (uint32_t)(__ffs((int)mk) - 1) >> 3;
                line_start[++o] = p + (uint32_t)k * 4 + b + 1;
                mk &= mk - 1;
            }
        }
        run += total;
    }
}

struct ParseArgs {
    const uint8_t* text;
    uint64_t n;                       // text bytes
    const unsigned long long* line_start;
    uint64_t n_lines;
    int unterminated;                 // the last line has no '\n' (and so keeps a trailing '\r', misc str::lines semantics)
    TokTable tb;
    tok::LineRec* recs;
    unsigned long long *s_al, *s_ops, *s_blk;   // [n_lines + 1] scan inputs: aligned?, CIGAR ops, sequence blocks
    TokStatus* st;
};

__device__ __forceinline__ void line_span(const ParseArgs& a, tok::Txt& x, uint64_t i, uint64_t& s, uint64_t& e) {
    s = a.line_start[i];
    if (i + 1 == a.n_lines && a.unterminated) { e = a.n; return; }
    e = a.line_start[i + 1] - 1;
    if (e > s && x.at(e - 1) == '\r') e--;
}

__global__ void __launch_bounds__(TK_LINE_THREADS) k_tok_parse(ParseArgs a) {
    __shared__ uint8_t s_nib[256];
    for (int k = threadIdx.x; k < 256; k += TK_LINE_THREADS) s_nib[k] = a.tb.nibtab[k];
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (i > a.n_lines) return;
    if (i == a.n_lines) { a.s_al[i] = 0; a.s_ops[i] = 0; a.s_blk[i] = 0; return; }
    tok::Txt x(a.text);
    uint64_t s, e;
    line_span(a, x, i, s, e);
    tok::LineRec r;
    const uint8_t kind = tok::parse_line(x, s, e, a.tb.ct, s_nib, r);
    r.kind = kind;
    a.recs[i] = r;
    const bool al = kind == tok::LK_ALIGNED;
    a.s_al[i] = al ? 1 : 0;
    a.s_ops[i] = al ? r.nops : 0;
    a.s_blk[i] = al ? tok::seq_blocks(r) : 0;
    if (kind == tok::LK_HOST) atomicMin(&a.st->first_bad, (unsigned long long)i);
    if (al && r.need8) a.st->need8 = 1;
}

struct EmitArgs {
    ParseArgs p;
    uint64_t aln_base, ops_base, blk_base;
    uint32_t *contig, *ref_start, *seq_off, *cigar_off, *nm, *cigar_ops;
    uint16_t *seq_len, *n_cigar;
    uint8_t *flags, *seq_pool;
    unsigned long long* name_pos;     // [alignments of this file] text offset of the QNAME
    uint32_t* name_len;
};

template <int BITS>
__global__ void __launch_bounds__(TK_LINE_THREADS) k_tok_emit(EmitArgs a) {
    __shared__ uint8_t s_nib[256];
    for (int k = threadIdx.x; k < 256; k += TK_LINE_THREADS) s_nib[k] = a.p.tb.nibtab[k];
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (i >= a.p.n_lines) return;
    const tok::LineRec r = a.p.recs[i];
    if (r.kind != tok::LK_ALIGNED) return;
    const uint64_t s = a.p.line_start[i];
    const uint64_t la = a.p.s_al[i], A = a.aln_base + la;
    const uint64_t co = a.ops_base + a.p.s_ops[i], bo = a.blk_base + a.p.s_blk[i];
    const bool star = r.flags & PP_FLAG_SEQSTAR;
    a.contig[A] = r.contig;
    a.ref_start[A] = r.ref_start;
    a.seq_off[A] = star ? 0u : (uint32_t)bo;
    a.seq_len[A] = (uint16_t)r.slen;
    a.cigar_off[A] = (uint32_t)co;
    a.n_cigar[A] = (uint16_t)r.nops;
    a.nm[A] = r.nm;
    a.flags[A] = r.flags;
    a.name_pos[la] = s;
    a.name_len[la] = r.name_len;
    tok::Txt x(a.p.text);
    tok::emit_cigar(x, s, r, a.cigar_ops + co);
    if (tok::emit_seq<BITS>(x, s, r, s_nib, a.seq_pool + bo * (BITS == 4 ? 16 : 32))) a.p.st->need8 = 1;
}

__global__ void __launch_bounds__(TK_LINE_THREADS) k_tok_heads(const uint8_t* __restrict__ text, uint64_t n_al, const unsigned long long* __restrict__ name_pos,
                                                               const uint32_t* __restrict__ name_len, uint32_t* __restrict__ head) {
    const uint64_t a = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (a >= n_al) return;
    tok::Txt x(text);
    head[a] = tok::group_head(x, a, 0, reinterpret_cast<const uint64_t*>(name_pos), name_len) ? 1u : 0u;
}

__global__ void __launch_bounds__(TK_LINE_THREADS) k_tok_groups(uint64_t n_al, const uint32_t* __restrict__ head, const uint32_t* __restrict__ rs, uint64_t read_base,
                                                                int careful, uint32_t* __restrict__ read_id, uint32_t* seq_off, uint16_t* seq_len, uint8_t* flags,
                                                                TokStatus* st) {
    const uint64_t a = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (a >= n_al) return;
    read_id[a] = (uint32_t)(read_base + rs[a] - 1);
    if (head[a] && !tok::close_group(a, n_al, head, careful != 0, seq_off, seq_len, flags)) st->group_err = 1;
}

// ---- BAM records (bam_rec.h): the image of the file stands in for the text, record offsets for line starts
struct BamArgs {
    ParseArgs p;
    const uint32_t* ref_contig;       // [n_ref + 1]
    uint32_t n_ref;
};

__global__ void __launch_bounds__(TK_LINE_THREADS) k_bam_parse(BamArgs a) {
    const uint64_t i = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (i > a.p.n_lines) return;
    if (i == a.p.n_lines) { a.p.s_al[i] = 0; a.p.s_ops[i] = 0; a.p.s_blk[i] = 0; return; }
    tok::Txt x(a.p.text);
    tok::LineRec r;
    uint8_t fault;
    const uint8_t kind = tok::parse_bam(x, a.p.line_start[i], a.ref_contig, a.n_ref, r, fault);
    a.p.recs[i] = r;
    const bool al = kind == tok::LK_ALIGNED;
    a.p.s_al[i] = al ? 1 : 0;
    a.p.s_ops[i] = al ? r.nops : 0;
    a.p.s_blk[i] = al ? tok::seq_blocks(r) : 0;
    if (kind == tok::LK_HOST) atomicMin(&a.p.st->first_bad, (unsigned long long)i);
}

template <int BITS>
__global__ void __launch_bounds__(TK_LINE_THREADS) k_bam_emit(EmitArgs a) {
    const uint64_t i = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (i >= a.p.n_lines) return;
    const tok::LineRec r = a.p.recs[i];
    if (r.kind != tok::LK_ALIGNED) return;
    const uint64_t s = a.p.line_start[i];
    const uint64_t la = a.p.s_al[i], A = a.aln_base + la;
    const uint64_t co = a.ops_base + a.p.s_ops[i], bo = a.blk_base + a.p.s_blk[i];
    const bool star = r.flags & PP_FLAG_SEQSTAR;
    a.contig[A] = r.contig;
    a.ref_start[A] = r.ref_start;
    a.seq_off[A] = star ? 0u : (uint32_t)bo;
    a.seq_len[A] = (uint16_t)r.slen;
    a.cigar_off[A] = (uint32_t)co;
    a.n_cigar[A] = (uint16_t)r.nops;
    a.nm[A] = r.nm;
    a.flags[A] = r.flags;
    a.name_pos[la] = s + tok::BAM_FIXED;          // read_name: k_tok_heads compares QNAMEs in the image as it does in text
    a.name_len[la] = r.name_len;
    tok::Txt x(a.p.text);
    tok::emit_bam_cigar(x, s, r, a.cigar_ops + co);
    if (tok::emit_bam_seq<BITS>(x, s, r, a.seq_pool + bo * (BITS == 4 ? 16 : 32))) a.p.st->need8 = 1;
}

}  // namespace

struct TokFilterBufs;

struct TokState {
    const pp_fasta* fasta = nullptr;
    bool careful = false, active = false;
    int seq_bits = 4;
    uint64_t aln_base = 0, ops_base = 0, blk_base = 0, read_base = 0;   // dataset under construction
    TokTable tb{};
    TokStatus* h_st = nullptr;            // pinned
    unsigned long long* h_tot = nullptr;  // pinned [4]
    TokStatus* d_st = nullptr;
    // file streaming
    uint8_t* pin[TK_READERS][2] = {};
    cudaStream_t rstream[TK_READERS] = {};
    cudaEvent_t rev[TK_READERS][2] = {};
    int readers = 0;                      // threads in use (pp_tok_set_readers, default from the core count)
    int ring = 0;                         // readers whose slots / stream exist
    // text buffers: one being tokenised, one being filled by the background upload of the next file
    DevBuf text[2];
    int next_buf = 0;
    uint64_t expect_total = 0;            // pp_tok_expect: bytes of all the files of this dataset (sizes the arrays once)
    struct Prefetch {
        std::thread th;
        bool active = false;
        std::string path;
        int buf = 0;
        uint64_t n = 0;
        uint8_t last = '\n';
        int rc = PP_OK;                   // PP_OK, PP_ERR_IO, PP_ERR_CUDA
        int cuda_err = 0;
        float ms = 0;
        uint64_t off = 0;                 // first byte of the file that is sent (pp_tok_set_ranges)
        bool strip = false;               // uploaded with QUAL replaced by "*" (polish only: filter reproduces lines verbatim)
        uint64_t sent = 0;                // bytes that crossed PCIe
    } pf;
    bool strip_qual = false;              // pp_tok_set_strip_qual (off by default: measured host-bound, see profiles/README.md)
    uint8_t* h_nl = nullptr;              // pinned '\n'
    DevBuf cub;
    TokFilterBufs* fbufs = nullptr;   // device buffers of the filter text path
    // pp_tok_set_ranges: this context tokenises one byte range of every file (multi-GPU ingestion); marks[f] = the dataset's
    // (alignments, ops, sequence blocks, reads) when file f started, marks.back() = now
    bool ranges_on = false;
    std::vector<uint64_t> range_off, range_len;
    struct Mark { uint64_t aln, ops, blk, reads; };
    std::vector<Mark> marks;
    // pp_tok_set_bam_range: file f of pp_tok_add_files is records [r0, r1) of an image the caller decoded (several contexts share it)
    struct BamIn { const pp::BamImage* im = nullptr; uint64_t r0 = 0, r1 = 0; };
    std::vector<BamIn> bam_in;
    // what the last pp_tok_add_files found per file: BAM or not, and for a BAM where the load's time went (host read, inflate and
    // record walk of bam.cpp - zero for an image the caller decoded - then the image and record offsets to HBM)
    struct BamPhase { bool bam = false; float read_ms = 0, inflate_ms = 0, walk_ms = 0, upload_ms = 0; };
    std::vector<BamPhase> phases;
    struct XState;                    // buffers of pp_tok_exchange_finish, kept between calls (no cudaMalloc in the steady state)
    XState* xs = nullptr;
    // pp_tok_set_shard: this context keeps one shard of the assembly
    bool shard_on = false, shard_unknown = false;
    DevBuf shard_map;                 // local_of[c] on the device
    uint32_t shard_n_total = 0;
    std::vector<uint64_t> shard_off;
    std::vector<uint8_t> shard_bases;
};

static void free_filter_bufs(TokFilterBufs* b);
static void free_xstate(TokState* T);

void pp_tok_release(pp_ctx* ctx) {
    TokState* T = ctx->tok;
    if (!T) return;
    if (T->fbufs) { free_filter_bufs(T->fbufs); T->fbufs = nullptr; }
    if (T->pf.active && T->pf.th.joinable()) T->pf.th.join();
    T->text[0].release(); T->text[1].release();
    for (int r = 0; r < TK_READERS; ++r) {
        for (int k = 0; k < 2; ++k) {
            if (T->pin[r][k]) cudaFreeHost(T->pin[r][k]);
            if (T->rev[r][k]) cudaEventDestroy(T->rev[r][k]);
        }
        if (T->rstream[r]) cudaStreamDestroy(T->rstream[r]);
    }
    if (T->h_st) cudaFreeHost(T->h_st);
    if (T->h_nl) cudaFreeHost(T->h_nl);
    if (T->h_tot) cudaFreeHost(T->h_tot);
    if (T->d_st) cudaFree(T->d_st);
    T->cub.release();
    T->shard_map.release();
    free_xstate(T);
    delete T;
    ctx->tok = nullptr;
}

static int tok_state(pp_ctx* ctx, TokState** out) {
    if (!ctx->tok) {
        TokState* T = new TokState();
        ctx->tok = T;
        CK(cudaHostAlloc((void**)&T->h_st, sizeof(TokStatus), cudaHostAllocDefault));
        CK(cudaHostAlloc((void**)&T->h_tot, 4 * sizeof(unsigned long long), cudaHostAllocDefault));
        CK(cudaMalloc((void**)&T->d_st, sizeof(TokStatus)));
        CK(cudaHostAlloc((void**)&T->h_nl, 64, cudaHostAllocDefault));
        T->h_nl[0] = '\n';
    }
    *out = ctx->tok;
    return PP_OK;
}

// Grows a dataset buffer keeping its first `keep` bytes (the alignments of the files tokenised so far).
static int ensure_keep(pp_ctx* ctx, int which, size_t bytes, size_t keep) {
    DevBuf& b = ctx->b[which];
    if (bytes <= b.cap) return PP_OK;
    if (keep == 0) { CK(b.ensure(bytes)); return PP_OK; }
    void* np = nullptr;
    const size_t want = bytes + bytes / 4 + 256;
    CK(cudaMalloc(&np, want));
    cudaError_t e = cudaMemcpyAsync(np, b.p, keep, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { cudaFree(np); CK(e); }
    cudaFree(b.p);
    b.p = np;
    b.cap = want;
    return PP_OK;
}

int pp_ctx_upload_contigs(pp_ctx* ctx, const pp_contigs* c);
int pp_ctx_commit_dataset(pp_ctx* ctx, uint64_t n_aln, uint64_t n_reads, uint64_t n_ops, uint64_t seq_bytes, uint32_t seq_bits);

extern "C" int pp_tok_begin(pp_ctx* ctx, const pp_fasta* fa, int careful, int seq_bits) {
    if (!ctx) return PP_ERR_ARG;
    if (!fa || (seq_bits != 4 && seq_bits != 8)) return ctx->fail(PP_ERR_ARG, "pp_tok_begin: null assembly or seq_bits not 4 / 8");
    CK(cudaSetDevice(ctx->device));
    TokState* T = nullptr;
    int rc = tok_state(ctx, &T);
    if (rc) return rc;
    ctx->have_ds = false;
    pp_contigs contigs;
    pp_fasta_view(fa, &contigs);
    if ((rc = pp_ctx_upload_contigs(ctx, &contigs))) return rc;
    tok::TableImage im;
    tok::build_table_image(fa->names, im);
    CK(ctx->b[B_TOKNAMES].ensure(im.bytes.size()));
    CK(cudaMemcpyAsync(ctx->b[B_TOKNAMES].p, im.bytes.data(), im.bytes.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));              // `im` is pageable and about to go away
    const uint8_t* base = ctx->b[B_TOKNAMES].as<uint8_t>();
    T->tb.ct = tok::table_view(im, base);
    T->tb.nibtab = base + im.o_nib;
    T->fasta = fa; T->careful = careful != 0; T->seq_bits = seq_bits;
    T->aln_base = T->ops_base = T->blk_base = T->read_base = 0;
    T->expect_total = 0;
    T->active = true;
    T->shard_on = false;
    T->ranges_on = false;
    T->marks.clear();
    T->bam_in.clear();
    return PP_OK;
}

int pp_tok_set_bam_range(pp_ctx* ctx, int file, const pp::BamImage* im, uint64_t r0, uint64_t r1) {
    TokState* T = ctx ? ctx->tok : nullptr;
    if (!T || !T->active || file < 0 || !im || r0 > r1 || r1 > im->rec.size()) return PP_ERR_ARG;
    if (T->bam_in.size() <= (size_t)file) T->bam_in.resize((size_t)file + 1);
    T->bam_in[(size_t)file] = {im, r0, r1};
    return PP_OK;
}

// Optional, after pp_tok_begin: the i-th path of pp_tok_add_files contributes only bytes [off[i], off[i] + len[i]) - a range that
// starts at a line start and ends behind a line end, cut between two read groups (the caller's job: host_api.cpp split_ranges).
// A range without alignments is fine (the file as a whole is the caller's to check).
extern "C" int pp_tok_set_ranges(pp_ctx* ctx, const uint64_t* off, const uint64_t* len, int n) {
    if (!ctx) return PP_ERR_ARG;
    TokState* T = ctx->tok;
    if (!T || !T->active) return ctx->fail(PP_ERR_ARG, "pp_tok_set_ranges: no pp_tok_begin");
    if (n < 0 || (n && (!off || !len))) return ctx->fail(PP_ERR_ARG, "pp_tok_set_ranges: null ranges");
    T->range_off.assign(off, off + n);
    T->range_len.assign(len, len + n);
    T->ranges_on = true;
    return PP_OK;
}

// Records of contigs this shard does not hold become ghosts (shard.cpp does the same on the host: contig 0, PP_FLAG_GHOST); the rest
// get the shard's contig numbers.
__global__ void k_shard_mark(uint32_t* __restrict__ contig, uint8_t* __restrict__ flags, uint64_t n_aln, const uint32_t* __restrict__ local_of,
                             uint32_t n_total, int takes_unknown) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_aln; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t c = contig[i];
        uint32_t l = 0xFFFFFFFFu;
        if (c == PP_CONTIG_UNKNOWN || c >= n_total) { if (takes_unknown) continue; }
        else l = local_of[c];
        if (l == 0xFFFFFFFFu) { contig[i] = 0; flags[i] |= PP_FLAG_GHOST; }
        else contig[i] = l;
    }
}

extern "C" int pp_tok_set_shard(pp_ctx* ctx, const uint32_t* local_of, uint32_t n_contigs_total, const pp_contigs* sc, int takes_unknown) {
    if (!ctx) return PP_ERR_ARG;
    TokState* T = ctx->tok;
    if (!T || !T->active) return ctx->fail(PP_ERR_ARG, "pp_tok_set_shard: no pp_tok_begin");
    if (!local_of || !sc || !sc->off || !sc->bases || sc->n_contigs == 0) return ctx->fail(PP_ERR_ARG, "pp_tok_set_shard: null or empty shard");
    for (uint32_t c = 0; c < n_contigs_total; ++c)
        if (local_of[c] != 0xFFFFFFFFu && local_of[c] >= sc->n_contigs) return ctx->fail(PP_ERR_ARG, "pp_tok_set_shard: local index outside the shard");
    CK(cudaSetDevice(ctx->device));
    CK(T->shard_map.ensure((size_t)n_contigs_total * 4 + 16));
    CK(cudaMemcpyAsync(T->shard_map.p, local_of, (size_t)n_contigs_total * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    T->shard_off.assign(sc->off, sc->off + sc->n_contigs + 1);
    T->shard_bases.assign(sc->bases, sc->bases + sc->off[sc->n_contigs]);
    T->shard_n_total = n_contigs_total;
    T->shard_unknown = takes_unknown != 0;
    T->shard_on = true;
    return PP_OK;
}

// Scratch of the per-line passes (one line = one SAM text line or one BAM record): line starts | line records | three scan arrays;
// the status is reset.
static int line_scratch(pp_ctx* ctx, TokState* T, const uint8_t* text, uint64_t n, uint64_t n_lines, ParseArgs& pa) {
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~size_t(255); return o; };
    const size_t o_ls = carve((n_lines + 2) * 8), o_rec = carve(n_lines * sizeof(tok::LineRec)), o_al = carve((n_lines + 1) * 8),
                 o_ops = carve((n_lines + 1) * 8), o_blk = carve((n_lines + 1) * 8);
    TRY_ALLOC(ctx->b[B_TOKTMP].ensure(off));
    uint8_t* tmp = ctx->b[B_TOKTMP].as<uint8_t>();
    pa.text = text; pa.n = n; pa.line_start = (unsigned long long*)(tmp + o_ls); pa.n_lines = n_lines; pa.unterminated = 0;
    pa.tb = T->tb; pa.recs = (tok::LineRec*)(tmp + o_rec);
    pa.s_al = (unsigned long long*)(tmp + o_al); pa.s_ops = (unsigned long long*)(tmp + o_ops); pa.s_blk = (unsigned long long*)(tmp + o_blk);
    pa.st = T->d_st;
    T->h_st->first_bad = ~0ull; T->h_st->need8 = 0; T->h_st->group_err = 0;
    CK(cudaMemcpyAsync(T->d_st, T->h_st, sizeof(TokStatus), cudaMemcpyHostToDevice, ctx->stream));
    return PP_OK;
}

// What the SAM and the BAM front ends share once the parse pass has run: the scans (alignment index, CIGAR-pool and sequence-pool
// offsets), the dataset arrays, the emit pass (`emit(ea, grid)` launches the front end's emit kernel), read groups, the SEQ="*"
// sources, and the commit of the dataset bases.
template <class Emit>
static int tok_emit_groups(pp_ctx* ctx, TokState* T, const ParseArgs& pa, bool part_of_file, uint32_t launches, pp_tok_stats* stats, Emit&& emit) {
    cudaStream_t s = ctx->stream;
    const uint8_t* text = pa.text;
    const uint64_t n = pa.n, n_lines = pa.n_lines;
    size_t cub_bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, pa.s_al, pa.s_al, (int64_t)(n_lines + 1)));
    CK(T->cub.ensure(cub_bytes + 256));
    for (unsigned long long* arr : {pa.s_al, pa.s_ops, pa.s_blk}) {
        size_t tb = T->cub.cap;
        CK(cub::DeviceScan::ExclusiveSum(T->cub.p, tb, arr, arr, (int64_t)(n_lines + 1), s));
    }
    CK(cudaMemcpyAsync(T->h_tot + 0, pa.s_al + n_lines, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(T->h_tot + 1, pa.s_ops + n_lines, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(T->h_tot + 2, pa.s_blk + n_lines, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(T->h_st, T->d_st, sizeof(TokStatus), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    launches += 3;
    const uint64_t n_al = T->h_tot[0], n_ops = T->h_tot[1], n_blk = T->h_tot[2];
    if (stats) stats->alignments = n_al;
    if (T->h_st->first_bad != ~0ull) return PP_TOK_HOST;
    if (n_al == 0) return part_of_file ? PP_OK : PP_TOK_HOST;      // alignment.rs:268-270
    if (T->aln_base + n_al >= 0xFFFFFFFFull - 4096 || T->ops_base + n_ops > 0xFFFFFFFFull || T->blk_base + n_blk > 0xFFFFFFFFull) return PP_TOK_HOST;

    // ---- dataset arrays (kept across files)
    const uint64_t A0 = T->aln_base, A1 = A0 + n_al;
    const size_t blk_bytes = T->seq_bits == 4 ? 16 : 32;
    // first file of a dataset whose total text size is known: size the arrays for all of it (no regrowth, no cudaFree later)
    double grow = 1.0;
    if (A0 == 0 && T->expect_total > n && n > 0) grow = std::min(64.0, 1.03 * (double)T->expect_total / (double)n);
    auto want = [&](uint64_t items, size_t each) { return (size_t)((double)items * grow) * each; };
    int rc;
    for (int w : {B_CONTIG, B_REFSTART, B_READID, B_SEQOFF, B_CIGOFF, B_NM})
        if ((rc = ensure_keep(ctx, w, std::max<size_t>(A1 * 4, want(n_al, 4)) + 64, A0 * 4))) return rc;
    for (int w : {B_SEQLEN, B_NCIG})
        if ((rc = ensure_keep(ctx, w, std::max<size_t>(A1 * 2, want(n_al, 2)) + 64, A0 * 2))) return rc;
    if ((rc = ensure_keep(ctx, B_FLAGS, std::max<size_t>(A1, want(n_al, 1)) + 64, A0))) return rc;
    if ((rc = ensure_keep(ctx, B_CIGOPS, std::max<size_t>((T->ops_base + n_ops) * 4, want(n_ops, 4)) + 64, T->ops_base * 4))) return rc;
    if ((rc = ensure_keep(ctx, B_SEQPOOL, std::max<size_t>((T->blk_base + n_blk) * blk_bytes, want(n_blk, blk_bytes)) + 256, T->blk_base * blk_bytes))) return rc;
    // per-alignment scratch of this file: QNAME position / length, group heads, their running count
    size_t off2 = 0;
    auto carve2 = [&](size_t bytes) { size_t o = off2; off2 += (bytes + 255) & ~size_t(255); return o; };
    const size_t o_np = carve2(n_al * 8), o_nl = carve2(n_al * 4), o_hd = carve2(n_al * 4), o_rs = carve2(n_al * 4);
    TRY_ALLOC(ctx->b[B_SCRATCH].ensure(off2));
    uint8_t* sc = ctx->b[B_SCRATCH].as<uint8_t>();

    EmitArgs ea;
    ea.p = pa; ea.aln_base = A0; ea.ops_base = T->ops_base; ea.blk_base = T->blk_base;
    ea.contig = ctx->b[B_CONTIG].as<uint32_t>(); ea.ref_start = ctx->b[B_REFSTART].as<uint32_t>(); ea.seq_off = ctx->b[B_SEQOFF].as<uint32_t>();
    ea.cigar_off = ctx->b[B_CIGOFF].as<uint32_t>(); ea.nm = ctx->b[B_NM].as<uint32_t>(); ea.cigar_ops = ctx->b[B_CIGOPS].as<uint32_t>();
    ea.seq_len = ctx->b[B_SEQLEN].as<uint16_t>(); ea.n_cigar = ctx->b[B_NCIG].as<uint16_t>();
    ea.flags = ctx->b[B_FLAGS].as<uint8_t>(); ea.seq_pool = ctx->b[B_SEQPOOL].as<uint8_t>();
    ea.name_pos = (unsigned long long*)(sc + o_np); ea.name_len = (uint32_t*)(sc + o_nl);
    emit(ea, (unsigned)((n_lines + TK_LINE_THREADS - 1) / TK_LINE_THREADS));
    uint32_t* head = (uint32_t*)(sc + o_hd);
    uint32_t* rs = (uint32_t*)(sc + o_rs);
    const unsigned aln_grid = (unsigned)((n_al + TK_LINE_THREADS - 1) / TK_LINE_THREADS);
    k_tok_heads<<<aln_grid, TK_LINE_THREADS, 0, s>>>(text, n_al, ea.name_pos, ea.name_len, head);
    CK(cub::DeviceScan::InclusiveSum(nullptr, cub_bytes, head, rs, (int64_t)n_al));
    CK(T->cub.ensure(cub_bytes + 256));
    {
        size_t tb = T->cub.cap;
        CK(cub::DeviceScan::InclusiveSum(T->cub.p, tb, head, rs, (int64_t)n_al, s));
    }
    k_tok_groups<<<aln_grid, TK_LINE_THREADS, 0, s>>>(n_al, head, rs, T->read_base, T->careful ? 1 : 0, ctx->b[B_READID].as<uint32_t>() + A0,
                                                       ea.seq_off + A0, ea.seq_len + A0, ea.flags + A0, T->d_st);
    uint32_t* h_reads = (uint32_t*)(T->h_tot + 3);
    CK(cudaMemcpyAsync(h_reads, rs + (n_al - 1), 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(T->h_st, T->d_st, sizeof(TokStatus), cudaMemcpyDeviceToHost, s));
    CK(cudaEventRecord(ctx->ev[1], s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    launches += 4;
    if (T->h_st->group_err) return PP_TOK_HOST;
    if (T->h_st->need8 && T->seq_bits == 4) return PP_TOK_NEED8;   // found while the bases were converted (k_tok_emit)
    const uint64_t n_reads = *h_reads;
    if (T->read_base + n_reads >= 0xFFFFFFFFull) return PP_TOK_HOST;
    T->aln_base = A1; T->ops_base += n_ops; T->blk_base += n_blk; T->read_base += n_reads;
    if (stats) {
        stats->reads = n_reads;
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
        stats->device_ms = ms;
        stats->launches = launches;
    }
    return PP_OK;
}


// The text is on the device (n bytes, zero padded).  Appends its alignments to the dataset under construction.
static int tok_process(pp_ctx* ctx, TokState* T, const uint8_t* text, uint64_t n, bool unterminated, pp_tok_stats* stats, bool part_of_file = false) {
    cudaStream_t s = ctx->stream;
    uint32_t launches = 0;
    CK(cudaEventRecord(ctx->ev[0], s));
    // ---- lines
    const uint64_t n16 = (n + 15) & ~15ull;
    const uint64_t n_tiles = (n16 + TK_TILE - 1) / TK_TILE;
    if (n_tiles >= 0x7FFFFFFFull) return PP_TOK_HOST;
    size_t cub_bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (int64_t)std::max<uint64_t>(n_tiles + 1, 1)));
    CK(T->cub.ensure(cub_bytes + 256));
    TRY_ALLOC(ctx->b[B_TOKLINE].ensure((n_tiles + 2) * 8));
    unsigned long long* tile_cnt = ctx->b[B_TOKLINE].as<unsigned long long>();
    uint64_t n_lines = 0;
    if (n_tiles) {
        CK(cudaMemsetAsync(tile_cnt + n_tiles, 0, 8, s));
        k_tok_count<<<(unsigned)n_tiles, TK_THREADS, 0, s>>>(text, n16, tile_cnt);
        size_t tb = T->cub.cap;
        CK(cub::DeviceScan::ExclusiveSum(T->cub.p, tb, tile_cnt, tile_cnt, (int64_t)(n_tiles + 1), s));
        CK(cudaMemcpyAsync(T->h_tot, tile_cnt + n_tiles, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        launches += 3;
        n_lines = T->h_tot[0] + (unterminated ? 1 : 0);
    }
    if (stats) stats->lines = n_lines;
    if (n_lines == 0) return part_of_file ? PP_OK : PP_TOK_HOST;   // "no alignments in <file>": the host packer words it (a byte range may be empty)
    if (n_lines >= 0xFFFFFFF0ull) return PP_TOK_HOST;

    ParseArgs pa;
    int rc = line_scratch(ctx, T, text, n, n_lines, pa);
    if (rc != PP_OK) return rc;
    pa.unterminated = unterminated ? 1 : 0;
    k_tok_index<<<(unsigned)n_tiles, TK_THREADS, 0, s>>>(text, n16, tile_cnt, const_cast<unsigned long long*>(pa.line_start));
    const unsigned line_grid = (unsigned)((n_lines + 1 + TK_LINE_THREADS - 1) / TK_LINE_THREADS);
    k_tok_parse<<<line_grid, TK_LINE_THREADS, 0, s>>>(pa);
    launches += 2;
    return tok_emit_groups(ctx, T, pa, part_of_file, launches, stats, [&](const EmitArgs& ea, unsigned grid) {
        if (T->seq_bits == 4) k_tok_emit<4><<<grid, TK_LINE_THREADS, 0, s>>>(ea);
        else k_tok_emit<8><<<grid, TK_LINE_THREADS, 0, s>>>(ea);
    });
}

static int text_buffer(pp_ctx* ctx, DevBuf& tb, uint64_t n) {
    CK(tb.ensure(n + 64));
    const uint64_t n16 = (n + 15) & ~15ull;
    CK(cudaMemsetAsync(tb.as<uint8_t>() + n, 0, (size_t)(n16 + 32 - n), ctx->stream));   // the copies never touch [n, ...)
    return PP_OK;
}

extern "C" int pp_tok_add_text(pp_ctx* ctx, const char* text, size_t len, pp_tok_stats* stats) {
    if (!ctx) return PP_ERR_ARG;
    TokState* T = ctx->tok;
    if (!T || !T->active) return ctx->fail(PP_ERR_ARG, "pp_tok_add_text: no pp_tok_begin");
    if (!text && len) return ctx->fail(PP_ERR_ARG, "pp_tok_add_text: null text");
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof *stats);
    if (T->pf.active) { if (T->pf.th.joinable()) T->pf.th.join(); T->pf.active = false; }
    DevBuf& tb = T->text[T->next_buf];
    T->next_buf ^= 1;
    int rc = text_buffer(ctx, tb, len);
    if (rc) return rc;
    const auto t0 = std::chrono::steady_clock::now();
    if (len) CK(cudaMemcpyAsync(tb.p, text, len, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const float h2d = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    rc = tok_process(ctx, T, tb.as<uint8_t>(), len, len > 0 && text[len - 1] != '\n', stats);
    if (stats) { stats->h2d_ms = h2d; stats->h2d_bytes = len; }
    if (rc != PP_OK) T->active = false;
    return rc;
}

// Streams a file into dst: T->readers host threads, each pread()s its slices into its two pinned slots and sends them on
// its own stream, so that page-cache reads, pinned staging and PCIe overlap.  Runs on the caller's thread or on the
// prefetch thread; touches neither ctx->err nor ctx->stream.  Returns PP_OK / PP_ERR_IO / PP_ERR_CUDA (+ *cuda_err).
static int upload_file(int device, TokState* T, uint8_t* dst, int fd, uint64_t n, uint8_t* last_byte, int* cuda_err, uint64_t foff = 0,
                       const uint8_t* mem = nullptr /* the bytes are in host memory (a BAM image), not in fd */) {
    const int R = T->readers;
    const uint64_t n_slices = (n + TK_SLOT - 1) / TK_SLOT;
    std::atomic<int> err{0};           // 1 = read error, 2 = CUDA error
    std::atomic<int> cerr{0};
    auto work = [&](int r) {
        if (cudaSetDevice(device) != cudaSuccess) { err = 2; return; }
        uint64_t k = 0;
        for (uint64_t sl = (uint64_t)r; sl < n_slices && !err; sl += (uint64_t)R, ++k) {
            const int slot = (int)(k & 1);
            if (k >= 2) {
                cudaError_t e = cudaEventSynchronize(T->rev[r][slot]);
                if (e != cudaSuccess) { cerr = (int)e; err = 2; return; }
            }
            const uint64_t o = sl * TK_SLOT, len = std::min<uint64_t>(TK_SLOT, n - o);
            uint64_t got = 0;
            if (mem) memcpy(T->pin[r][slot], mem + o, (size_t)len), got = len;
            while (got < len) {
                const ssize_t g = pread(fd, T->pin[r][slot] + got, (size_t)(len - got), (off_t)(foff + o + got));
                if (g <= 0) { err = 1; return; }
                got += (uint64_t)g;
            }
            if (o + len == n) *last_byte = T->pin[r][slot][len - 1];
            cudaError_t e = cudaMemcpyAsync(dst + o, T->pin[r][slot], (size_t)len, cudaMemcpyHostToDevice, T->rstream[r]);
            if (e == cudaSuccess) e = cudaEventRecord(T->rev[r][slot], T->rstream[r]);
            if (e != cudaSuccess) { cerr = (int)e; err = 2; return; }
        }
        cudaError_t e = cudaStreamSynchronize(T->rstream[r]);
        if (e != cudaSuccess) { cerr = (int)e; err = 2; }
    };
    std::vector<std::thread> th;
    for (int r = 1; r < R; ++r) th.emplace_back(work, r);
    work(0);
    for (auto& t : th) t.join();
    *cuda_err = cerr.load();
    return err == 1 ? PP_ERR_IO : err == 2 ? PP_ERR_CUDA : PP_OK;
}

constexpr int PP_UPLOAD_LONG_LINE = 100;   // internal: a line longer than TK_LOOK, upload the file verbatim instead

// The same for `polish`, with less on the wire: every reader owns the LINES that start in its nominal slice, replaces their
// QUAL by "*" while staging them (tok_strip.h: 45 % of a bwa-mem line, never read on this path) and sends the shorter text
// to the lines' original offset; the freed tail of the slice becomes one '@' comment line on the device ('@', blanks
// written by a memset, '\n'), which every parser of this path skips (alignment.rs:241-242).  Offsets, and therefore the
// independence of the readers, stay as they are.  A file whose last line is unterminated keeps its last slice verbatim.
static int upload_file_stripped(int device, TokState* T, uint8_t* dst, int fd, uint64_t n, uint8_t* last_byte, int* cuda_err, uint64_t* sent) {
    const int R = T->readers;
    const uint64_t S = TK_SLOT - TK_LOOK;
    const uint64_t n_slices = (n + S - 1) / S;
    std::atomic<int> err{0}, cerr{0};              // 1 read error, 2 CUDA error, 3 long line
    std::atomic<unsigned long long> bytes{0};
    // the lines are read through a private mapping of the file where that works (no copy before the strip), else pread
    const uint8_t* map = nullptr;
    {
        void* m = n ? mmap(nullptr, (size_t)n, PROT_READ, MAP_PRIVATE, fd, 0) : MAP_FAILED;
        if (m != MAP_FAILED) { map = (const uint8_t*)m; madvise(m, (size_t)n, MADV_SEQUENTIAL); }
    }
    auto work = [&](int r) {
        if (cudaSetDevice(device) != cudaSuccess) { err = 2; return; }
        std::vector<uint8_t> rawbuf(map ? 16 : TK_SLOT + 16);
        uint64_t j = 0;
        for (uint64_t k = (uint64_t)r; k < n_slices && !err; k += (uint64_t)R) {
            const uint64_t o = k * S, e = std::min<uint64_t>(n, o + S);
            const uint64_t rd0 = k ? o - 1 : 0, rd1 = std::min<uint64_t>(n, e + TK_LOOK - 1);
            const uint8_t* raw = map ? map + rd0 : rawbuf.data();
            if (!map) {
                uint64_t got = 0;
                while (got < rd1 - rd0) {
                    const ssize_t g = pread(fd, rawbuf.data() + got, (size_t)(rd1 - rd0 - got), (off_t)(rd0 + got));
                    if (g <= 0) { err = 1; return; }
                    got += (uint64_t)g;
                }
            }
            // the slot is needed before the lines are staged into it
            const int slot = (int)(j & 1);
            if (j >= 2) {
                cudaError_t ce = cudaEventSynchronize(T->rev[r][slot]);
                if (ce != cudaSuccess) { cerr = (int)ce; err = 2; return; }
            }
            uint8_t* pin = T->pin[r][slot];
            const tok::SliceOut so = tok::strip_slice(raw, rd0, rd1, k, e, n, pin);
            if (so.status == 3) { err = 3; return; }
            if (so.status == 1) continue;                          // one long line covers the whole slice: an earlier slice owns it
            ++j;
            if (so.ends_file) *last_byte = so.last;
            const uint64_t a = so.a, b = so.b, c = so.c, gap = (b - a) - c;
            cudaError_t ce = cudaSuccess;
            if (gap == 0) {
                ce = cudaMemcpyAsync(dst + a, pin, (size_t)c, cudaMemcpyHostToDevice, T->rstream[r]);
            } else if (gap == 1) {
                pin[c] = '\n';                                      // an empty line
                ce = cudaMemcpyAsync(dst + a, pin, (size_t)c + 1, cudaMemcpyHostToDevice, T->rstream[r]);
            } else {
                pin[c] = '@';                                       // a comment line of gap bytes
                ce = cudaMemcpyAsync(dst + a, pin, (size_t)c + 1, cudaMemcpyHostToDevice, T->rstream[r]);
                if (ce == cudaSuccess && gap > 2) ce = cudaMemsetAsync(dst + a + c + 1, ' ', (size_t)(gap - 2), T->rstream[r]);
                if (ce == cudaSuccess) ce = cudaMemcpyAsync(dst + b - 1, T->h_nl, 1, cudaMemcpyHostToDevice, T->rstream[r]);
            }
            if (ce == cudaSuccess) ce = cudaEventRecord(T->rev[r][slot], T->rstream[r]);
            if (ce != cudaSuccess) { cerr = (int)ce; err = 2; return; }
            bytes += c + (gap ? 2 : 0);
        }
        cudaError_t ce = cudaStreamSynchronize(T->rstream[r]);
        if (ce != cudaSuccess) { cerr = (int)ce; err = 2; }
    };
    std::vector<std::thread> th;
    for (int r = 1; r < R; ++r) th.emplace_back(work, r);
    work(0);
    for (auto& t : th) t.join();
    if (map) munmap((void*)map, (size_t)n);
    *cuda_err = cerr.load();
    *sent = bytes.load();
    if (err == 3) {                                   // let the copies that were issued finish before the verbatim upload reuses the slots
        for (int r = 0; r < R; ++r) cudaStreamSynchronize(T->rstream[r]);
        return PP_UPLOAD_LONG_LINE;
    }
    return err == 1 ? PP_ERR_IO : err == 2 ? PP_ERR_CUDA : PP_OK;
}

static int ring_ready(pp_ctx* ctx, TokState* T) {
    if (T->readers <= 0) {
        const unsigned hw = std::thread::hardware_concurrency();
        T->readers = (int)std::min<unsigned>(TK_READERS, std::max<unsigned>(2, hw / 4));
    }
    for (int r = T->ring; r < T->readers; ++r) {
        CK(cudaStreamCreateWithFlags(&T->rstream[r], cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            CK(cudaHostAlloc((void**)&T->pin[r][k], TK_SLOT, cudaHostAllocDefault));
            CK(cudaEventCreateWithFlags(&T->rev[r][k], cudaEventDisableTiming));
        }
        T->ring = r + 1;
    }
    return PP_OK;
}

// Starts streaming `path` into the next text buffer on a background thread.  PP_OK, PP_TOK_HOST (not a plain readable
// file) or an error.
static int prefetch_start(pp_ctx* ctx, TokState* T, const char* path, bool strip, int range = -1) {
    struct stat sb;
    if (stat(path, &sb) != 0 || !S_ISREG(sb.st_mode)) return PP_TOK_HOST;   // pipes, devices: never opened here (the host path streams them once)
    const int fd = open(path, O_RDONLY);
    if (fd < 0 || fstat(fd, &sb) != 0 || !S_ISREG(sb.st_mode)) {
        if (fd >= 0) close(fd);
        return PP_TOK_HOST;
    }
    uint64_t n = (uint64_t)sb.st_size, foff = 0;
    if (range >= 0) {
        if ((size_t)range >= T->range_off.size() || T->range_off[range] + T->range_len[range] > n) { close(fd); return PP_TOK_HOST; }
        foff = T->range_off[range]; n = T->range_len[range];
        strip = false;                                           // (the stripping upload works on whole files)
    }
    const int buf = T->next_buf;
    int rc = ring_ready(ctx, T);
    if (rc != PP_OK) { close(fd); return rc; }
    if (T->text[buf].cap < n + 64) {
        // The text, its line index / records and the arrays built from it must fit beside what is already resident; a file too
        // large for that goes through the host parser (which needs no device memory for text).
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || (double)free_b + (double)T->text[buf].cap < 2.6 * (double)n + (256 << 20)) {
            cudaGetLastError();
            close(fd);
            return PP_TOK_HOST;
        }
    }
    rc = text_buffer(ctx, T->text[buf], n);
    if (rc != PP_OK) { cudaGetLastError(); close(fd); return PP_TOK_HOST; }
    T->next_buf ^= 1;
    TokState::Prefetch& pf = T->pf;
    pf.active = true; pf.path = path; pf.buf = buf; pf.n = n; pf.last = '\n'; pf.rc = PP_OK; pf.cuda_err = 0; pf.ms = 0;
    pf.strip = strip && T->strip_qual; pf.sent = 0; pf.off = foff;
    uint8_t* dst = T->text[buf].as<uint8_t>();
    const int device = ctx->device;
    pf.th = std::thread([T, dst, fd, n, device, foff] {
        TokState::Prefetch& q = T->pf;
        const auto t0 = std::chrono::steady_clock::now();
        if (n && q.strip) {
            q.rc = upload_file_stripped(device, T, dst, fd, n, &q.last, &q.cuda_err, &q.sent);
            if (q.rc == PP_UPLOAD_LONG_LINE) q.strip = false;
        }
        if (n && !q.strip) { q.rc = upload_file(device, T, dst, fd, n, &q.last, &q.cuda_err, foff); q.sent = n; }
        close(fd);
        q.ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    });
    return PP_OK;
}

// Waits for the text of `path` (starting its upload now if nobody asked for it before).
static int prefetch_wait(pp_ctx* ctx, TokState* T, const char* path, bool strip, int range = -1) {
    TokState::Prefetch& pf = T->pf;
    const bool other_range = range >= 0 && (size_t)range < T->range_off.size() && (pf.off != T->range_off[range] || pf.n != T->range_len[range]);
    if (pf.active && (pf.path != path || (pf.strip && !strip) || other_range || (range < 0 && pf.off != 0))) {   // (text without QUAL is no use to `filter`)                       // something else was prefetched: let it finish, drop it
        if (pf.th.joinable()) pf.th.join();
        pf.active = false;
    }
    if (!pf.active) {
        const int rc = prefetch_start(ctx, T, path, strip, range);
        if (rc != PP_OK) return rc;
    }
    if (pf.th.joinable()) pf.th.join();
    pf.active = false;
    if (pf.rc == PP_ERR_IO) return PP_TOK_HOST;               // the host path reports unreadable files
    if (pf.rc == PP_ERR_CUDA) return ctx->fail_cuda((cudaError_t)pf.cuda_err, "SAM text upload", __FILE__, __LINE__);
    return PP_OK;
}

extern "C" int pp_tok_prefetch(pp_ctx* ctx, const char* path) {
    if (!ctx || !path) return PP_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    TokState* T = nullptr;
    int rc = tok_state(ctx, &T);
    if (rc) return rc;
    if (T->pf.active) return PP_OK;                            // one outstanding upload at a time
    if (pp::is_bam(path)) return PP_OK;                        // a BAM is inflated on the host first (tok_add_bam)
    rc = prefetch_start(ctx, T, path, true);
    return rc == PP_TOK_HOST ? PP_OK : rc;                     // pp_tok_add_file(s) will say so
}

extern "C" int pp_tok_expect(pp_ctx* ctx, uint64_t total_text_bytes) {
    if (!ctx) return PP_ERR_ARG;
    TokState* T = nullptr;
    int rc = tok_state(ctx, &T);
    if (rc) return rc;
    T->expect_total = total_text_bytes;
    return PP_OK;
}

// Records [r0, r1) of a BAM image -> appended to the dataset under construction.  The image crosses PCIe through the reader slots,
// then k_bam_parse / k_bam_emit decode it in place.  `next` (may be null): the next file, which starts streaming in once the slots
// are free again (a SAM file: the caller has classified it).  host_ms: what reading, inflating and walking the file took (part of
// h2d_ms); *upload_ms: the image and the record offsets to HBM.
static int tok_add_bam(pp_ctx* ctx, TokState* T, const pp::BamImage& im, uint64_t r0, uint64_t r1, pp_tok_stats* stats, float host_ms,
                       const char* next, int next_range, float* upload_ms) {
    cudaStream_t s = ctx->stream;
    const uint64_t n_rec = r1 - r0;
    if (stats) stats->lines = n_rec;
    if (!im.device_ok) return PP_TOK_HOST;
    if (n_rec == 0) return T->ranges_on ? PP_OK : PP_TOK_HOST;         // "no alignments in <file>": the host packer words it
    if (n_rec >= 0xFFFFFFF0ull) return PP_TOK_HOST;
    const uint64_t b0 = im.rec[r0], b1 = r1 < im.rec.size() ? im.rec[r1] : im.size, n = b1 - b0;
    int rc = ring_ready(ctx, T);
    if (rc != PP_OK) return rc;
    const int buf = T->next_buf;
    T->next_buf ^= 1;
    DevBuf& tb = T->text[buf];
    if (tb.cap < n + 64) {                                             // the same room as a SAM text of this size needs
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || (double)free_b + (double)tb.cap < 2.6 * (double)n + (256 << 20)) {
            cudaGetLastError();
            return PP_TOK_HOST;
        }
    }
    rc = text_buffer(ctx, tb, n);
    if (rc != PP_OK) { cudaGetLastError(); return PP_TOK_HOST; }
    const auto t0 = std::chrono::steady_clock::now();
    uint8_t last = 0;
    int cerr = 0;
    rc = upload_file(ctx->device, T, tb.as<uint8_t>(), -1, n, &last, &cerr, 0, im.data.p + b0);
    if (rc == PP_ERR_CUDA) return ctx->fail_cuda((cudaError_t)cerr, "BAM image upload", __FILE__, __LINE__);
    ParseArgs pa;
    if ((rc = line_scratch(ctx, T, tb.as<uint8_t>(), n, n_rec, pa)) != PP_OK) return rc;
    {
        std::vector<unsigned long long> off((size_t)n_rec);
        for (uint64_t k = 0; k < n_rec; ++k) off[(size_t)k] = im.rec[r0 + k] - b0;
        CK(cudaMemcpyAsync(const_cast<unsigned long long*>(pa.line_start), off.data(), (size_t)n_rec * 8, cudaMemcpyHostToDevice, s));
        TRY_ALLOC(ctx->b[B_TOKLINE].ensure(im.ref_contig.size() * 4 + 16));
        CK(cudaMemcpyAsync(ctx->b[B_TOKLINE].p, im.ref_contig.data(), im.ref_contig.size() * 4, cudaMemcpyHostToDevice, s));
        CK(cudaStreamSynchronize(s));                                   // (pageable sources)
    }
    *upload_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    const float h2d = host_ms + *upload_ms;
    if (next && (rc = prefetch_start(ctx, T, next, true, next_range)) < 0) return rc;
    CK(cudaEventRecord(ctx->ev[0], s));
    BamArgs ba;
    ba.p = pa;
    ba.ref_contig = ctx->b[B_TOKLINE].as<uint32_t>();
    ba.n_ref = (uint32_t)im.ref_names.size();
    k_bam_parse<<<(unsigned)((n_rec + 1 + TK_LINE_THREADS - 1) / TK_LINE_THREADS), TK_LINE_THREADS, 0, s>>>(ba);
    rc = tok_emit_groups(ctx, T, pa, T->ranges_on, 1, stats, [&](const EmitArgs& ea, unsigned grid) {
        if (T->seq_bits == 4) k_bam_emit<4><<<grid, TK_LINE_THREADS, 0, s>>>(ea);
        else k_bam_emit<8><<<grid, TK_LINE_THREADS, 0, s>>>(ea);
    });
    if (stats) { stats->h2d_ms = h2d; stats->h2d_bytes = n + n_rec * 8; }
    return rc;
}

extern "C" int pp_tok_add_files(pp_ctx* ctx, const char* const* paths, int n_paths, pp_tok_stats* stats) {
    if (!ctx) return PP_ERR_ARG;
    TokState* T = ctx->tok;
    if (!T || !T->active) return ctx->fail(PP_ERR_ARG, "pp_tok_add_file: no pp_tok_begin");
    if (!paths || n_paths < 0) return ctx->fail(PP_ERR_ARG, "pp_tok_add_file: null paths");
    CK(cudaSetDevice(ctx->device));
    if (stats) memset(stats, 0, sizeof(pp_tok_stats) * (size_t)n_paths);
    if (T->ranges_on && T->range_off.size() != (size_t)n_paths) return ctx->fail(PP_ERR_ARG, "pp_tok_add_files: as many paths as pp_tok_set_ranges ranges");
    const bool ranges = T->ranges_on;
    // every input is classified once, here: a range of an image the caller decoded, a BAM file, or SAM text
    T->phases.assign((size_t)n_paths, TokState::BamPhase());
    for (int i = 0; i < n_paths; ++i) {
        if (!paths[i]) return ctx->fail(PP_ERR_ARG, "pp_tok_add_file: null path");
        T->phases[(size_t)i].bam = ((size_t)i < T->bam_in.size() && T->bam_in[(size_t)i].im) || pp::is_bam(paths[i]);
    }
    auto is_sam = [&](int j) { return j < n_paths && !T->phases[(size_t)j].bam; };
    for (int i = 0; i < n_paths; ++i) {
        T->marks.push_back({T->aln_base, T->ops_base, T->blk_base, T->read_base});
        TokState::BamPhase& ph = T->phases[(size_t)i];
        const TokState::BamIn* shared = (size_t)i < T->bam_in.size() && T->bam_in[(size_t)i].im ? &T->bam_in[(size_t)i] : nullptr;
        if (ph.bam) {
            if (T->pf.active) { if (T->pf.th.joinable()) T->pf.th.join(); T->pf.active = false; }   // (the reader slots are needed)
            if (!shared && ranges) { T->active = false; return PP_TOK_HOST; }                      // byte ranges are SAM-only
            pp::BamImage own;
            std::string err;
            if (!shared && pp::bam_load(paths[i], T->fasta, own, err) != PP_OK) { T->active = false; return PP_TOK_HOST; }   // the host words it
            const pp::BamImage& im = shared ? *shared->im : own;
            if (!shared) { ph.read_ms = im.read_ms; ph.inflate_ms = im.inflate_ms; ph.walk_ms = im.walk_ms; }
            const char* next = is_sam(i + 1) ? paths[i + 1] : nullptr;
            const int brc = tok_add_bam(ctx, T, im, shared ? shared->r0 : 0, shared ? shared->r1 : im.rec.size(), stats ? stats + i : nullptr,
                                        ph.read_ms + ph.inflate_ms + ph.walk_ms, next, ranges ? i + 1 : -1, &ph.upload_ms);
            if (brc != PP_OK) { T->active = false; return brc; }
            continue;
        }
        int rc = prefetch_wait(ctx, T, paths[i], true, ranges ? i : -1);
        if (rc != PP_OK) { T->active = false; return rc; }
        const int buf = T->pf.buf;
        const uint64_t n = T->pf.n;
        const bool unterminated = n > 0 && T->pf.last != '\n';
        const float h2d = T->pf.ms;
        const uint64_t h2d_bytes = T->pf.sent;
        if (is_sam(i + 1)) {                                    // the next file streams in while this one is tokenised
            rc = prefetch_start(ctx, T, paths[i + 1], true, ranges ? i + 1 : -1);
            if (rc < 0) { T->active = false; return rc; }
        }
        rc = tok_process(ctx, T, T->text[buf].as<uint8_t>(), n, unterminated, stats ? stats + i : nullptr, ranges);
        if (stats) { stats[i].h2d_ms = h2d; stats[i].h2d_bytes = h2d_bytes; }
        if (rc != PP_OK) { T->active = false; return rc; }
    }
    T->marks.push_back({T->aln_base, T->ops_base, T->blk_base, T->read_base});
    return PP_OK;
}

int pp_tok_bam_phases(pp_ctx* ctx, int file, float* read_ms, float* inflate_ms, float* walk_ms, float* upload_ms) {
    TokState* T = ctx ? ctx->tok : nullptr;
    if (!T || file < 0 || (size_t)file >= T->phases.size() || !T->phases[(size_t)file].bam) return 0;
    const TokState::BamPhase& ph = T->phases[(size_t)file];
    *read_ms = ph.read_ms; *inflate_ms = ph.inflate_ms; *walk_ms = ph.walk_ms; *upload_ms = ph.upload_ms;
    return 1;
}

extern "C" int pp_tok_add_file(pp_ctx* ctx, const char* path, pp_tok_stats* stats) {
    return pp_tok_add_files(ctx, &path, 1, stats);
}

extern "C" int pp_set_parser(pp_ctx* ctx, int mode) {
    if (!ctx || mode < 0 || mode > 1) return PP_ERR_ARG;
    ctx->parser = mode;
    return PP_OK;
}
extern "C" int pp_get_parser(const pp_ctx* ctx) { return ctx ? ctx->parser : 0; }

// Host threads that stream a SAM file into the device (0 = from the core count: a quarter of them, 2..16).
extern "C" int pp_tok_set_readers(pp_ctx* ctx, int n) {
    if (!ctx || n < 0 || n > TK_READERS) return PP_ERR_ARG;
    TokState* T = nullptr;
    int rc = tok_state(ctx, &T);
    if (rc) return rc;
    T->readers = n;
    return PP_OK;
}

// 1: pp_tok_add_file(s) / pp_tok_prefetch send the text without its QUAL column; 0 (default): byte for byte.
extern "C" int pp_tok_set_strip_qual(pp_ctx* ctx, int on) {
    if (!ctx) return PP_ERR_ARG;
    TokState* T = nullptr;
    int rc = tok_state(ctx, &T);
    if (rc) return rc;
    T->strip_qual = on != 0;
    return PP_OK;
}

extern "C" int pp_tok_finish(pp_ctx* ctx) {
    if (!ctx) return PP_ERR_ARG;
    TokState* T = ctx->tok;
    if (!T || !T->active) return ctx->fail(PP_ERR_ARG, "pp_tok_finish: no tokenised text");
    T->active = false;
    if (T->shard_on) {
        T->shard_on = false;
        CK(cudaSetDevice(ctx->device));
        if (T->aln_base)
            k_shard_mark<<<(uint32_t)std::min<uint64_t>((T->aln_base + 255) / 256, (uint64_t)ctx->sm_count * 32), 256, 0, ctx->stream>>>(
                ctx->b[B_CONTIG].as<uint32_t>(), ctx->b[B_FLAGS].as<uint8_t>(), T->aln_base, T->shard_map.as<uint32_t>(), T->shard_n_total,
                T->shard_unknown ? 1 : 0);
        pp_contigs sc;
        sc.n_contigs = (uint32_t)T->shard_off.size() - 1; sc.off = T->shard_off.data(); sc.bases = T->shard_bases.data();
        int rc = pp_ctx_upload_contigs(ctx, &sc);           // the shard's contigs are the draft from here on
        if (rc != PP_OK) return rc;
        CK(cudaStreamSynchronize(ctx->stream));             // (pageable sources)
        CK(cudaGetLastError());
        std::vector<uint8_t>().swap(T->shard_bases);
    }
    return pp_ctx_commit_dataset(ctx, T->aln_base, T->read_base, T->ops_base, T->blk_base * (T->seq_bits == 4 ? 16 : 32), (uint32_t)T->seq_bits);
}

// =====================================================================================================================
// Multi-GPU ingestion without the host in the middle (SURVEY.md §8e at file level).  Every context has tokenised ITS byte range of
// every SAM file (pp_tok_set_ranges; the ranges are cut between read groups).  pp_tok_exchange_finish then gives every GPU its
// shard: a read group goes - whole, so that k still spans contigs - to every GPU that owns a contig one of its records lies on.
// Per source GPU g and destination o: a bit mask per group (k_x_touch), four exclusive scans over the kept records (records, CIGAR
// ops, sequence blocks, groups), a compaction into staging arrays with every offset already renumbered for its place in o's
// dataset (k_x_pack*), and device-to-device copies (cudaMemcpyPeerAsync, NVLink where the box has it) into o's arrays at
// [file f][range g] - global SAM order is (file, range, line), which is what the ordered depth needs.  The host only adds up
// the piece sizes.  Then pp_tok_set_shard / pp_tok_finish on every GPU: foreign records become ghosts, the shard is binned.
// =====================================================================================================================
#define X_MAX_FILES 64
struct XPlan {                       // per (source, destination): where the pieces of each file go
    uint32_t n_files;
    uint32_t mark_aln[X_MAX_FILES + 1];                                   // first local record of file f
    uint32_t dst_aln[X_MAX_FILES], dst_ops[X_MAX_FILES], dst_blk[X_MAX_FILES], dst_grp[X_MAX_FILES];   // position in the destination's dataset
};

__global__ void k_x_touch(const uint32_t* __restrict__ contig, const uint32_t* __restrict__ read_id, uint64_t n, const uint32_t* __restrict__ owner,
                          uint32_t n_total, uint32_t read0, uint32_t* __restrict__ touch) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t c = contig[i];
        const uint32_t o = (c == PP_CONTIG_UNKNOWN || c >= n_total) ? 0u : owner[c];      // unknown RNAMEs stay with shard 0 (shard.cpp)
        atomicOr(&touch[read_id[i] - read0], 1u << o);
    }
}

// kept record -> (1, its ops, its own sequence blocks, 1 if it starts a group); element n is the scans' total slot
__global__ void k_x_flags(const uint32_t* __restrict__ read_id, const uint16_t* __restrict__ n_cigar, const uint16_t* __restrict__ seq_len,
                          const uint8_t* __restrict__ flags, uint64_t n, uint32_t read0, const uint32_t* __restrict__ touch, uint32_t dest,
                          uint32_t* __restrict__ f_rec, uint32_t* __restrict__ f_ops, uint32_t* __restrict__ f_blk, uint32_t* __restrict__ f_grp) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i <= n; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t r = 0, o = 0, b = 0, g = 0;
        if (i < n && ((touch[read_id[i] - read0] >> dest) & 1u)) {
            r = 1; o = n_cigar[i];
            if (!(flags[i] & (PP_FLAG_SEQSTAR | PP_FLAG_NOSEQ))) b = ((uint32_t)seq_len[i] + PP_SEQ_BLOCK - 1) / PP_SEQ_BLOCK;
            g = (i == 0 || read_id[i] != read_id[i - 1]) ? 1u : 0u;
        }
        f_rec[i] = r; f_ops[i] = o; f_blk[i] = b; f_grp[i] = g;
    }
}

__global__ void k_x_marks(const uint32_t* __restrict__ s_rec, const uint32_t* __restrict__ s_ops, const uint32_t* __restrict__ s_blk,
                          const uint32_t* __restrict__ s_grp, XPlan plan, uint32_t* __restrict__ out) {
    const uint32_t f = threadIdx.x;
    if (f <= plan.n_files) {
        const uint32_t i = plan.mark_aln[f];
        out[4 * f + 0] = s_rec[i]; out[4 * f + 1] = s_ops[i]; out[4 * f + 2] = s_blk[i]; out[4 * f + 3] = s_grp[i];
    }
}

struct XArrays {
    const uint32_t *contig, *ref_start, *read_id, *seq_off, *cigar_off, *nm, *cigar_ops;
    const uint16_t *seq_len, *n_cigar;
    const uint8_t *flags, *seq_pool;
};
struct XStage {
    uint32_t *contig, *ref_start, *read_id, *seq_off, *cigar_off, *nm, *cigar_ops;
    uint16_t *seq_len, *n_cigar;
    uint8_t *flags, *seq_pool;
};

// records that own their sequence: where its first block goes (indexed by the OLD block offset, local to this source)
__global__ void k_x_blockmap(XArrays a, uint64_t n, uint32_t blk0, const uint32_t* __restrict__ s_rec_flag, const uint32_t* __restrict__ s_rec,
                             const uint32_t* __restrict__ s_blk, uint32_t* __restrict__ blockmap) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        if (s_rec[i + 1] == s_rec[i]) continue;                                        // not kept
        if (a.flags[i] & (PP_FLAG_SEQSTAR | PP_FLAG_NOSEQ)) continue;
        blockmap[a.seq_off[i] - blk0] = s_blk[i];
    }
}

__global__ void k_x_pack(XArrays a, XStage st, uint64_t n, uint32_t blk0, uint32_t blk_bytes, XPlan plan, const uint32_t* __restrict__ s_rec,
                         const uint32_t* __restrict__ s_ops, const uint32_t* __restrict__ s_blk, const uint32_t* __restrict__ s_grp,
                         const uint32_t* __restrict__ blockmap, const uint32_t* __restrict__ marks /* scans at the file starts */) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t j = s_rec[i];
        if (s_rec[i + 1] == j) continue;                                               // not kept
        uint32_t f = 0;
        while (f + 1 < plan.n_files && i >= plan.mark_aln[f + 1]) ++f;
        const uint32_t m_ops = marks[4 * f + 1], m_blk = marks[4 * f + 2], m_grp = marks[4 * f + 3];
        const uint8_t fl = a.flags[i];
        const bool starts = (i == 0 || a.read_id[i] != a.read_id[i - 1]);
        st.contig[j] = a.contig[i]; st.ref_start[j] = a.ref_start[i]; st.nm[j] = a.nm[i];
        st.seq_len[j] = a.seq_len[i]; st.n_cigar[j] = a.n_cigar[i]; st.flags[j] = fl;
        st.read_id[j] = plan.dst_grp[f] + (s_grp[i] + (starts ? 1u : 0u) - 1u - m_grp);
        st.cigar_off[j] = plan.dst_ops[f] + (s_ops[i] - m_ops);
        uint32_t so = 0;
        if (!(fl & PP_FLAG_NOSEQ)) so = plan.dst_blk[f] + (blockmap[a.seq_off[i] - blk0] - m_blk);
        st.seq_off[j] = so;
        const uint32_t nc = a.n_cigar[i], co = a.cigar_off[i];
        for (uint32_t t = 0; t < nc; ++t) st.cigar_ops[s_ops[i] + t] = a.cigar_ops[co + t];
    }
}

// the sequence blocks of kept owners, 16 bytes per thread
__global__ void k_x_pack_seq(XArrays a, XStage st, uint64_t n, uint32_t blk_bytes, const uint32_t* __restrict__ s_rec, const uint32_t* __restrict__ s_blk) {
    const uint32_t per = blk_bytes / 16;
    for (uint64_t i = blockIdx.x * (uint64_t)(blockDim.x / 8) + threadIdx.x / 8; i < n; i += (uint64_t)gridDim.x * (blockDim.x / 8)) {
        if (s_rec[i + 1] == s_rec[i]) continue;
        const uint32_t nb = s_blk[i + 1] - s_blk[i];                                   // 0 for records without their own sequence
        if (!nb) continue;
        const uint4* src = reinterpret_cast<const uint4*>(a.seq_pool + (size_t)a.seq_off[i] * blk_bytes);
        uint4* dst = reinterpret_cast<uint4*>(st.seq_pool + (size_t)s_blk[i] * blk_bytes);
        for (uint32_t q = threadIdx.x & 7; q < nb * per; q += 8) dst[q] = src[q];
    }
}

struct TokState::XState {            // one context's tokenised ranges, moved out of the dataset buffers
    DevBuf b[11];                    // B_CONTIG .. B_SEQPOOL, in the enum's order
    DevBuf stage[11], touch, fl[4], sc[4], blockmap, marks, cubtmp;
    uint64_t n = 0, ops = 0, blk = 0, reads = 0;
    std::vector<TokState::Mark> mk;
    DevBuf d_owner;
    uint32_t* h_marks = nullptr;     // pinned
    void release() { for (auto& x : b) x.release(); for (auto& x : stage) x.release(); touch.release(); for (auto& x : fl) x.release();
                     for (auto& x : sc) x.release(); blockmap.release(); marks.release(); cubtmp.release(); d_owner.release();
                     if (h_marks) cudaFreeHost(h_marks); h_marks = nullptr; }
};
static void free_xstate(TokState* T) { if (T->xs) { T->xs->release(); delete T->xs; T->xs = nullptr; } }
namespace {
typedef TokState::XState XSource;
const int X_BUFS[11] = {B_CONTIG, B_REFSTART, B_READID, B_SEQOFF, B_SEQLEN, B_CIGOFF, B_NCIG, B_NM, B_FLAGS, B_CIGOPS, B_SEQPOOL};
}

#define XCK(ctx_, x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { rc = (ctx_)->fail_cuda(e_, #x, __FILE__, __LINE__); goto done; } } while (0)

extern "C" int pp_tok_exchange_finish(pp_ctx* const* ctxs, int n_ctx, const uint32_t* owner, uint32_t n_total, const uint32_t* const* local_of,
                                      const pp_contigs* shard_contigs, uint64_t* n_aln_total) {
    if (!ctxs || n_ctx < 1 || !owner || !local_of || !shard_contigs) return PP_ERR_ARG;
    if (n_ctx > 32) return PP_TOK_HOST;                                                // (one bit per destination in a group's mask: the host sharder takes over)
    pp_ctx* c0 = ctxs[0];
    int rc = PP_OK;
    std::vector<XSource*> src((size_t)n_ctx, nullptr);
    const int seq_bits = c0->tok ? c0->tok->seq_bits : 4;
    const uint32_t blk_bytes = seq_bits == 4 ? 16 : 32;
    size_t n_files = 0;
    // counts[g][o][f][4]: what source g sends destination o out of file f
    std::vector<uint32_t> counts;
    uint64_t total_aln = 0;
    // ---- the tokenised arrays leave the dataset buffers (those will receive the shard)
    for (int g = 0; g < n_ctx; ++g) {
        pp_ctx* ctx = ctxs[g];
        TokState* T = ctx->tok;
        if (!T || !T->active || T->marks.size() < 2 || T->seq_bits != seq_bits) { rc = c0->fail(PP_ERR_ARG, "pp_tok_exchange_finish: a context without tokenised ranges"); goto done; }
        if (g == 0) n_files = T->marks.size() - 1;
        if (T->marks.size() - 1 != n_files || n_files > X_MAX_FILES) { rc = PP_TOK_HOST; goto done; }
        if (!T->xs) T->xs = new XSource();
        src[g] = T->xs;
        XSource& S = *src[g];
        S.n = T->aln_base; S.ops = T->ops_base; S.blk = T->blk_base; S.reads = T->read_base; S.mk = T->marks;
        for (int k = 0; k < 11; ++k) std::swap(S.b[k], ctx->b[X_BUFS[k]]);
        total_aln += S.n;
    }
    counts.assign((size_t)n_ctx * n_ctx * n_files * 4, 0);
    for (int g = 0; g < n_ctx; ++g) {
        XCK(ctxs[g], cudaSetDevice(ctxs[g]->device));
        if (!src[g]->h_marks) XCK(ctxs[g], cudaHostAlloc((void**)&src[g]->h_marks, (X_MAX_FILES + 1) * 4 * sizeof(uint32_t), cudaHostAllocDefault));
        for (int o = 0; o < n_ctx; ++o)                                                // NVLink between the GPUs where the box has it
            if (ctxs[o]->device != ctxs[g]->device) {
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, ctxs[g]->device, ctxs[o]->device) == cudaSuccess && can) cudaDeviceEnablePeerAccess(ctxs[o]->device, 0);
                cudaGetLastError();                                                    // (already enabled is fine)
            }
    }

    for (int pass = 0; pass < 2; ++pass) {
        // pass 0: sizes of every piece; (host: where every piece goes, destination arrays); pass 1: pack and send
        std::vector<std::vector<XPlan>> plans;
        if (pass == 1) {
            plans.assign((size_t)n_ctx, std::vector<XPlan>((size_t)n_ctx));
            for (int o = 0; o < n_ctx; ++o) {
                uint64_t at[4] = {0, 0, 0, 0};
                for (size_t f = 0; f < n_files; ++f)
                    for (int g = 0; g < n_ctx; ++g) {
                        XPlan& P = plans[g][o];
                        P.dst_aln[f] = (uint32_t)at[0]; P.dst_ops[f] = (uint32_t)at[1]; P.dst_blk[f] = (uint32_t)at[2]; P.dst_grp[f] = (uint32_t)at[3];
                        const uint32_t* c = &counts[(((size_t)g * n_ctx + o) * n_files + f) * 4];
                        for (int k = 0; k < 4; ++k) at[k] += c[k];
                    }
                if (at[0] >= 0x7FFFFFFFull - 4096 || at[1] > 0xFFFFFFFFull || at[2] > 0xFFFFFFFFull || at[3] >= 0xFFFFFFFFull) { rc = PP_TOK_HOST; goto done; }
                pp_ctx* ctx = ctxs[o];
                XCK(ctx, cudaSetDevice(ctx->device));
                const size_t each[11] = {4, 4, 4, 4, 2, 4, 2, 4, 1, 4, blk_bytes};
                const uint64_t cnt[11] = {at[0], at[0], at[0], at[0], at[0], at[0], at[0], at[0], at[0], at[1], at[2]};
                for (int k = 0; k < 11; ++k) XCK(ctx, ctx->b[X_BUFS[k]].ensure((size_t)cnt[k] * each[k] + 256));
                TokState* T = ctx->tok;
                T->aln_base = at[0]; T->ops_base = at[1]; T->blk_base = at[2]; T->read_base = at[3];
            }
        }
        // every source GPU works through its destinations on its own stream, driven by its own host thread
        auto per_source = [&](int g) -> int {
            pp_ctx* ctx = ctxs[g];
            XSource& S = *src[g];
            cudaStream_t st = ctx->stream;
            uint32_t* hm = S.h_marks;
            CK(cudaSetDevice(ctx->device));
            const uint64_t n = S.n;
            const uint32_t read0 = 0, blk0 = 0;
            const unsigned grid = (unsigned)std::min<uint64_t>((n + 256) / 256 + 1, (uint64_t)ctx->sm_count * 32);
            XArrays A{S.b[0].as<uint32_t>(), S.b[1].as<uint32_t>(), S.b[2].as<uint32_t>(), S.b[3].as<uint32_t>(), S.b[5].as<uint32_t>(), S.b[7].as<uint32_t>(),
                      S.b[9].as<uint32_t>(), S.b[4].as<uint16_t>(), S.b[6].as<uint16_t>(), S.b[8].as<uint8_t>(), S.b[10].as<uint8_t>()};
            const size_t each[11] = {4, 4, 4, 4, 2, 4, 2, 4, 1, 4, blk_bytes};
            if (pass == 0) {
                CK(S.d_owner.ensure((size_t)n_total * 4 + 16));
                CK(cudaMemcpyAsync(S.d_owner.p, owner, (size_t)n_total * 4, cudaMemcpyHostToDevice, st));
                CK(S.touch.ensure((size_t)S.reads * 4 + 16));
                CK(cudaMemsetAsync(S.touch.p, 0, (size_t)S.reads * 4 + 16, st));
                for (int k = 0; k < 4; ++k) { CK(S.fl[k].ensure((n + 2) * 4)); CK(S.sc[k].ensure((n + 2) * 4)); }
                CK(S.marks.ensure((X_MAX_FILES + 1) * 16));
                size_t tb = 0;
                CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, (const uint32_t*)nullptr, (uint32_t*)nullptr, (int64_t)(n + 1), st));
                CK(S.cubtmp.ensure(tb + 256));
                if (n) k_x_touch<<<grid, 256, 0, st>>>(A.contig, A.read_id, n, S.d_owner.as<uint32_t>(), n_total, read0, S.touch.as<uint32_t>());
            } else {
                const uint64_t cnt[11] = {n, n, n, n, n, n, n, n, n, S.ops, S.blk};
                for (int k = 0; k < 11; ++k) CK(S.stage[k].ensure((size_t)cnt[k] * each[k] + 256));
                CK(S.blockmap.ensure((size_t)S.blk * 4 + 16));
            }
            XPlan base;
            memset(&base, 0, sizeof base);
            base.n_files = (uint32_t)n_files;
            for (size_t f = 0; f <= n_files; ++f) base.mark_aln[f] = (uint32_t)S.mk[f].aln;
            for (int oo = 0; oo < n_ctx; ++oo) {
                const int o = (g + oo) % n_ctx;                                        // (the sources start on different destinations)
                uint32_t* fl[4] = {S.fl[0].as<uint32_t>(), S.fl[1].as<uint32_t>(), S.fl[2].as<uint32_t>(), S.fl[3].as<uint32_t>()};
                uint32_t* sc[4] = {S.sc[0].as<uint32_t>(), S.sc[1].as<uint32_t>(), S.sc[2].as<uint32_t>(), S.sc[3].as<uint32_t>()};
                k_x_flags<<<grid, 256, 0, st>>>(A.read_id, A.n_cigar, A.seq_len, A.flags, n, read0, S.touch.as<uint32_t>(), (uint32_t)o, fl[0], fl[1], fl[2], fl[3]);
                for (int k = 0; k < 4; ++k) {
                    size_t tb = S.cubtmp.cap;
                    CK(cub::DeviceScan::ExclusiveSum(S.cubtmp.p, tb, fl[k], sc[k], (int64_t)(n + 1), st));
                }
                XPlan P = pass == 1 ? plans[g][o] : base;
                P.n_files = base.n_files;
                memcpy(P.mark_aln, base.mark_aln, sizeof base.mark_aln);
                k_x_marks<<<1, X_MAX_FILES + 1, 0, st>>>(sc[0], sc[1], sc[2], sc[3], P, S.marks.as<uint32_t>());
                if (pass == 1 && n) {
                    XStage Z{S.stage[0].as<uint32_t>(), S.stage[1].as<uint32_t>(), S.stage[2].as<uint32_t>(), S.stage[3].as<uint32_t>(), S.stage[5].as<uint32_t>(),
                             S.stage[7].as<uint32_t>(), S.stage[9].as<uint32_t>(), S.stage[4].as<uint16_t>(), S.stage[6].as<uint16_t>(), S.stage[8].as<uint8_t>(),
                             S.stage[10].as<uint8_t>()};
                    k_x_blockmap<<<grid, 256, 0, st>>>(A, n, blk0, fl[0], sc[0], sc[2], S.blockmap.as<uint32_t>());
                    k_x_pack<<<grid, 256, 0, st>>>(A, Z, n, blk0, blk_bytes, P, sc[0], sc[1], sc[2], sc[3], S.blockmap.as<uint32_t>(), S.marks.as<uint32_t>());
                    k_x_pack_seq<<<(unsigned)std::min<uint64_t>((n + 31) / 32 + 1, (uint64_t)ctx->sm_count * 64), 256, 0, st>>>(A, Z, n, blk_bytes, sc[0], sc[2]);
                }
                CK(cudaMemcpyAsync(hm, S.marks.p, (n_files + 1) * 16, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));
                if (pass == 0) {
                    for (size_t f = 0; f < n_files; ++f)
                        for (int k = 0; k < 4; ++k)
                            counts[(((size_t)g * n_ctx + o) * n_files + f) * 4 + k] = hm[4 * (f + 1) + k] - hm[4 * f + k];
                    continue;
                }
                // the pieces travel: file f's kept records are one contiguous run of the staging arrays
                pp_ctx* dctx = ctxs[o];
                for (size_t f = 0; f < n_files; ++f) {
                    const uint32_t* m0 = hm + 4 * f;
                    const uint32_t* m1 = hm + 4 * (f + 1);
                    for (int k = 0; k < 11; ++k) {
                        const int q = k == 9 ? 1 : k == 10 ? 2 : 0;                   // which scan measures this array
                        const uint64_t from = m0[q], cntk = (uint64_t)m1[q] - m0[q];
                        const uint64_t to = q == 0 ? P.dst_aln[f] : q == 1 ? P.dst_ops[f] : P.dst_blk[f];
                        if (!cntk) continue;
                        uint8_t* dst = dctx->b[X_BUFS[k]].as<uint8_t>() + (size_t)to * each[k];
                        const uint8_t* sp = S.stage[k].as<uint8_t>() + (size_t)from * each[k];
                        if (dctx->device == ctx->device) CK(cudaMemcpyAsync(dst, sp, (size_t)cntk * each[k], cudaMemcpyDeviceToDevice, st));
                        else CK(cudaMemcpyPeerAsync(dst, dctx->device, sp, ctx->device, (size_t)cntk * each[k], st));
                    }
                }
                CK(cudaStreamSynchronize(st));                                         // (the staging arrays are reused for the next destination)
            }
            return PP_OK;
        };
        std::vector<int> prc((size_t)n_ctx, PP_OK);
        {
            std::vector<std::thread> th;
            for (int g = 1; g < n_ctx; ++g) th.emplace_back([&, g] { prc[(size_t)g] = per_source(g); });
            prc[0] = per_source(0);
            for (auto& t : th) t.join();
        }
        for (int g = 0; g < n_ctx; ++g)
            if (prc[(size_t)g] != PP_OK) { rc = prc[(size_t)g]; if (ctxs[g] != c0) c0->err = ctxs[g]->err; goto done; }
    }
    // ---- every GPU holds its groups in global SAM order: ghosts, the shard's contigs, binning
    for (int o = 0; o < n_ctx && rc == PP_OK; ++o) {
        pp_ctx* ctx = ctxs[o];
        if (cudaSetDevice(ctx->device) != cudaSuccess) { rc = PP_ERR_CUDA; break; }
        rc = pp_tok_set_shard(ctx, local_of[o], n_total, &shard_contigs[o], o == 0);
        if (rc == PP_OK) rc = pp_tok_finish(ctx);
        if (rc != PP_OK && ctx != c0) c0->err = ctx->err;
    }
    if (n_aln_total) *n_aln_total = total_aln;
done:
    for (int g = 0; g < n_ctx; ++g) {
        // (the buffers stay with the context: the range arrays that were swapped out are the spare capacity of the next call)
        if (rc != PP_OK && ctxs[g]->tok) ctxs[g]->tok->active = false;
    }
    return rc;
}

// ---- the resident dataset, read back (tests compare it with the host packer's arrays)
extern "C" int pp_dataset_sizes(pp_ctx* ctx, pp_alignments* out) {
    if (!ctx || !out) return PP_ERR_ARG;
    if (!ctx->have_ds) return ctx->fail(PP_ERR_ARG, "pp_dataset_sizes: no resident dataset");
    memset(out, 0, sizeof *out);
    out->n_aln = ctx->n_aln; out->n_reads = ctx->n_reads; out->n_cigar_ops = ctx->n_ops; out->seq_pool_bytes = ctx->seq_bytes;
    out->seq_bits = ctx->seq_bits;
    return PP_OK;
}

extern "C" int pp_dataset_download(pp_ctx* ctx, const pp_alignments* into) {
    if (!ctx || !into) return PP_ERR_ARG;
    if (!ctx->have_ds) return ctx->fail(PP_ERR_ARG, "pp_dataset_download: no resident dataset");
    if (into->n_aln != ctx->n_aln || into->n_cigar_ops != ctx->n_ops || into->seq_pool_bytes != ctx->seq_bytes)
        return ctx->fail(PP_ERR_ARG, "pp_dataset_download: sizes differ from pp_dataset_sizes");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const size_t n = (size_t)ctx->n_aln;
    auto get = [&](const void* dst, int which, size_t bytes) -> cudaError_t {
        if (!dst || !bytes) return cudaSuccess;
        return cudaMemcpyAsync(const_cast<void*>(dst), ctx->b[which].p, bytes, cudaMemcpyDeviceToHost, s);
    };
    CK(get(into->contig, B_CONTIG, n * 4)); CK(get(into->ref_start, B_REFSTART, n * 4)); CK(get(into->read_id, B_READID, n * 4));
    CK(get(into->seq_off, B_SEQOFF, n * 4)); CK(get(into->seq_len, B_SEQLEN, n * 2)); CK(get(into->cigar_off, B_CIGOFF, n * 4));
    CK(get(into->n_cigar, B_NCIG, n * 2)); CK(get(into->nm, B_NM, n * 4)); CK(get(into->flags, B_FLAGS, n));
    CK(get(into->cigar_ops, B_CIGOPS, (size_t)ctx->n_ops * 4)); CK(get(into->seq_pool, B_SEQPOOL, (size_t)ctx->seq_bytes));
    CK(cudaStreamSynchronize(s));
    return PP_OK;
}

// =====================================================================================================================
// `polypolish filter` on SAM text in HBM (SURVEY.md §8f-2): both files are streamed in, parsed (Alignment::new_quick,
// alignment.rs:102-128), their QNAMEs and RNAMEs interned in one device hash table (the reference's
// HashMap<String, Vec<Alignment>> keys, filter.rs:110-145), the filter proper runs on the arrays where they are
// (filter_kernels.cu), and the output SAM text (filter_sam, filter.rs:296-349: every line verbatim, "\tZP:Z:fail" appended to
// failing aligned records, '\n' line ends) is assembled on the device and streamed back into the output files.
// Anything unusual (a line the quick parse rejects, a file without alignments, a 64-bit hash collision between different
// strings, a size limit) answers PP_TOK_HOST and filter_pack.cpp does the job on the host, with the reference's messages.
// =====================================================================================================================
#include "filter_dev.h"

namespace {

struct FileDev {                       // one SAM file on the device
    const uint8_t* text;
    uint64_t n, n_lines;
    int unterminated;
    const unsigned long long* line_start;   // [n_lines + 1]
    tok::FLineRec* recs;                    // [n_lines]
    unsigned long long* s_al;               // [n_lines + 1] exclusive scan of "aligned"
    uint32_t *name_slot, *ref_slot;         // [n_lines] interned ids (aligned lines)
};

struct InternTable {
    unsigned long long* key;           // [cap] 0 = empty
    unsigned long long* rep;           // [cap] smallest (kind << 62 | file << 40 | line) that claimed the slot
    uint32_t mask;
};

struct FStatus {
    unsigned long long first_bad[2];   // per file: smallest line index the quick parse leaves to the host
    unsigned int collision;            // different strings with one 64-bit key, or a full table
    unsigned int pad;
};

__device__ __forceinline__ void fline_span(const FileDev& f, tok::Txt& x, uint64_t i, uint64_t& s, uint64_t& e) {
    s = f.line_start[i];
    if (i + 1 == f.n_lines && f.unterminated) { e = f.n; return; }
    e = f.line_start[i + 1] - 1;
    if (e > s && x.at(e - 1) == '\r') e--;
}

__global__ void __launch_bounds__(TK_LINE_THREADS) k_ftok_parse(FileDev f, int which, FStatus* st) {
    const uint64_t i = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (i > f.n_lines) return;
    if (i == f.n_lines) { f.s_al[i] = 0; return; }
    tok::Txt x(f.text);
    uint64_t s, e;
    fline_span(f, x, i, s, e);
    tok::FLineRec r;
    const uint8_t kind = tok::parse_line_quick(x, s, e, r);
    r.kind = kind;
    f.recs[i] = r;
    f.s_al[i] = kind == tok::FK_ALIGNED ? 1 : 0;
    if (kind == tok::FK_HOST) atomicMin(&st->first_bad[which], (unsigned long long)i);
}

constexpr unsigned long long REF_DOMAIN = 0x9E3779B97F4A7C15ull;

// Claims the slot of `key` (insert-only linear probing: a key sits in the first slot of its probe sequence that was empty
// when it arrived, and slots never empty again, so every later arrival of the same key finds it).
__device__ __forceinline__ uint32_t intern(const InternTable& t, unsigned long long key, unsigned long long who, FStatus* st) {
    if (key == 0) key = 1;
    uint32_t sl = (uint32_t)(key ^ (key >> 32)) & t.mask;
    for (uint32_t probes = 0; probes <= t.mask; ++probes, sl = (sl + 1) & t.mask) {
        unsigned long long cur = t.key[sl];
        if (cur == 0) cur = atomicCAS(&t.key[sl], 0ull, key);
        if (cur == 0 || cur == key) {
            if (t.rep[sl] > who) atomicMin(&t.rep[sl], who);
            return sl;
        }
    }
    st->collision = 1;                 // table full
    return 0;
}

__global__ void __launch_bounds__(TK_LINE_THREADS) k_ftok_intern(FileDev f, int which, InternTable t, FStatus* st) {
    const uint64_t i = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (i >= f.n_lines) return;
    const tok::FLineRec r = f.recs[i];
    if (r.kind != tok::FK_ALIGNED) return;
    const unsigned long long who = ((unsigned long long)which << 40) | i;
    f.name_slot[i] = intern(t, r.name_hash, who, st);
    f.ref_slot[i] = intern(t, r.ref_hash ^ REF_DOMAIN, (1ull << 62) | who, st);
}

// Every record confirms, byte by byte, that the string that owns its slot is its own string.
__global__ void __launch_bounds__(TK_LINE_THREADS) k_ftok_verify(FileDev f0, FileDev f1, int which, InternTable t, FStatus* st) {
    const FileDev& f = which ? f1 : f0;
    const uint64_t i = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (i >= f.n_lines) return;
    const tok::FLineRec r = f.recs[i];
    if (r.kind != tok::FK_ALIGNED) return;
    const uint64_t s = f.line_start[i];
    tok::Txt x(f.text);
    for (int kind = 0; kind < 2; ++kind) {
        const unsigned long long rep = t.rep[kind ? f.ref_slot[i] : f.name_slot[i]];
        const int rk = (int)(rep >> 62), rf = (int)((rep >> 40) & 1);
        const uint64_t rl = rep & ((1ull << 40) - 1);
        bool same = rk == kind;
        if (same) {
            const FileDev& g = rf ? f1 : f0;
            const tok::FLineRec q = g.recs[rl];
            const uint64_t qs = g.line_start[rl];
            tok::Txt y(g.text);
            if (kind == 0) same = q.name_len == r.name_len && tok::same_bytes(x, s, y, qs, r.name_len);
            else same = q.ref_len == r.ref_len && tok::same_bytes(x, s + r.ref_rel, y, qs + q.ref_rel, r.ref_len);
        }
        if (!same) st->collision = 1;
    }
}

struct MateOut { uint32_t *name_id, *contig, *ref_start, *ref_end; uint8_t* flags; };

__global__ void __launch_bounds__(TK_LINE_THREADS) k_ftok_emit(FileDev f, MateOut m) {
    const uint64_t i = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (i >= f.n_lines) return;
    const tok::FLineRec r = f.recs[i];
    if (r.kind != tok::FK_ALIGNED) return;
    const uint64_t a = f.s_al[i];
    m.name_id[a] = f.name_slot[i];
    m.contig[a] = f.ref_slot[i];
    m.ref_start[a] = r.ref_start;
    m.ref_end[a] = r.ref_end;
    m.flags[a] = r.rev;
}

// filter_sam (filter.rs:296-349): bytes of every output line.
__global__ void __launch_bounds__(TK_LINE_THREADS) k_ftok_outlen(FileDev f, const uint8_t* __restrict__ pass, unsigned long long* __restrict__ out_off) {
    const uint64_t i = (uint64_t)blockIdx.x * TK_LINE_THREADS + threadIdx.x;
    if (i > f.n_lines) return;
    if (i == f.n_lines) { out_off[i] = 0; return; }
    tok::Txt x(f.text);
    uint64_t s, e;
    fline_span(f, x, i, s, e);
    const bool fail = f.recs[i].kind == tok::FK_ALIGNED && !pass[f.s_al[i]];
    out_off[i] = (e - s) + 1 + (fail ? 10 : 0);
}

// One warp per line: the line's bytes, the tag for failing records, '\n'.
__global__ void __launch_bounds__(256) k_ftok_copy(FileDev f, const uint8_t* __restrict__ pass, const unsigned long long* __restrict__ out_off,
                                                   uint8_t* __restrict__ out) {
    const uint64_t i = ((uint64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31;
    if (i >= f.n_lines) return;
    uint64_t s = f.line_start[i], e;
    if (i + 1 == f.n_lines && f.unterminated) e = f.n;
    else { e = f.line_start[i + 1] - 1; if (e > s && f.text[e - 1] == '\r') e--; }
    const bool fail = f.recs[i].kind == tok::FK_ALIGNED && !pass[f.s_al[i]];
    uint8_t* d = out + out_off[i];
    const uint64_t len = e - s;
    for (uint64_t k = lane; k < len; k += 32) d[k] = f.text[s + k];
    if (fail) { if (lane < 10) d[len + lane] = (uint8_t)"\tZP:Z:fail"[lane]; }
    if (lane == 0) d[len + (fail ? 10 : 0)] = '\n';
}

}  // namespace

// Streams n device bytes into fd (the mirror image of upload_file): each thread copies its slices into its pinned slots and
// from there into the file.  `map` is the file mapped MAP_SHARED (page faults of different threads proceed in parallel,
// whereas write()s to one file serialise on its inode lock: 3 GB/s on tmpfs whatever the thread count); when the mapping
// could not be made, pwrite() is used.  PP_OK / PP_ERR_IO / PP_ERR_CUDA.
static int download_file(int device, TokState* T, const uint8_t* src, int fd, uint8_t* map, uint64_t n, int* cuda_err) {
    const int R = T->readers;
    const uint64_t n_slices = (n + TK_SLOT - 1) / TK_SLOT;
    std::atomic<int> err{0}, cerr{0};
    auto work = [&](int r) {
        if (cudaSetDevice(device) != cudaSuccess) { err = 2; return; }
        uint64_t k = 0, prev_o = 0, prev_len = 0;
        bool have_prev = false;
        auto flush_prev = [&](int slot) -> bool {
            cudaError_t e = cudaEventSynchronize(T->rev[r][slot]);
            if (e != cudaSuccess) { cerr = (int)e; err = 2; return false; }
            if (map) { memcpy(map + prev_o, T->pin[r][slot], (size_t)prev_len); return true; }
            uint64_t put = 0;
            while (put < prev_len) {
                const ssize_t g = pwrite(fd, T->pin[r][slot] + put, (size_t)(prev_len - put), (off_t)(prev_o + put));
                if (g <= 0) { err = 1; return false; }
                put += (uint64_t)g;
            }
            return true;
        };
        for (uint64_t sl = (uint64_t)r; sl < n_slices && !err; sl += (uint64_t)R, ++k) {
            const int slot = (int)(k & 1);
            const uint64_t o = sl * TK_SLOT, len = std::min<uint64_t>(TK_SLOT, n - o);
            cudaError_t e = cudaMemcpyAsync(T->pin[r][slot], src + o, (size_t)len, cudaMemcpyDeviceToHost, T->rstream[r]);
            if (e == cudaSuccess) e = cudaEventRecord(T->rev[r][slot], T->rstream[r]);
            if (e != cudaSuccess) { cerr = (int)e; err = 2; return; }
            if (have_prev && !flush_prev(slot ^ 1)) return;
            prev_o = o; prev_len = len; have_prev = true;
        }
        if (have_prev && !err) flush_prev((int)((k - 1) & 1));
    };
    std::vector<std::thread> th;
    for (int r = 1; r < R; ++r) th.emplace_back(work, r);
    work(0);
    for (auto& t : th) t.join();
    *cuda_err = cerr.load();
    return err == 1 ? PP_ERR_IO : err == 2 ? PP_ERR_CUDA : PP_OK;
}

// The same bytes to a descriptor that only takes sequential writes (pipe, FIFO, character device): one thread, two pinned slots,
// the copy of slice i+1 in flight while slice i is written.  PP_OK / PP_ERR_IO / PP_ERR_CUDA.
static int download_stream(int device, TokState* T, const uint8_t* src, int fd, uint64_t n, int* cuda_err) {
    if (cudaSetDevice(device) != cudaSuccess) return PP_ERR_CUDA;
    const uint64_t n_slices = (n + TK_SLOT - 1) / TK_SLOT;
    auto put_all = [&](const uint8_t* p, uint64_t len) {
        uint64_t put = 0;
        while (put < len) {
            const ssize_t g = write(fd, p + put, (size_t)(len - put));
            if (g < 0 && errno == EINTR) continue;
            if (g <= 0) return false;
            put += (uint64_t)g;
        }
        return true;
    };
    uint64_t prev_len = 0;
    for (uint64_t sl = 0; sl <= n_slices; ++sl) {
        const int slot = (int)(sl & 1);
        if (sl < n_slices) {
            const uint64_t o = sl * TK_SLOT, len = std::min<uint64_t>(TK_SLOT, n - o);
            cudaError_t e = cudaMemcpyAsync(T->pin[0][slot], src + o, (size_t)len, cudaMemcpyDeviceToHost, T->rstream[0]);
            if (e == cudaSuccess) e = cudaEventRecord(T->rev[0][slot], T->rstream[0]);
            if (e != cudaSuccess) { *cuda_err = (int)e; return PP_ERR_CUDA; }
        }
        if (sl > 0) {
            const cudaError_t e = cudaEventSynchronize(T->rev[0][slot ^ 1]);
            if (e != cudaSuccess) { *cuda_err = (int)e; return PP_ERR_CUDA; }
            if (!put_all(T->pin[0][slot ^ 1], prev_len)) return PP_ERR_IO;
        }
        if (sl < n_slices) prev_len = std::min<uint64_t>(TK_SLOT, n - sl * TK_SLOT);
    }
    return PP_OK;
}

// Line index + quick parse of one file whose text is on the device.  Fills fd; PP_OK / PP_TOK_HOST / error.
static int ftok_lines(pp_ctx* ctx, TokState* T, int which, const uint8_t* text, uint64_t n, bool unterminated, DevBuf& lines, DevBuf& tmp, FStatus* d_st,
                      FileDev* fd, uint32_t* launches) {
    cudaStream_t s = ctx->stream;
    const uint64_t n16 = (n + 15) & ~15ull;
    const uint64_t n_tiles = (n16 + TK_TILE - 1) / TK_TILE;
    if (n_tiles == 0 || n_tiles >= 0x7FFFFFFFull) return PP_TOK_HOST;
    size_t cub_bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (int64_t)(n_tiles + 1)));
    CK(T->cub.ensure(cub_bytes + 256));
    TRY_ALLOC(ctx->b[B_TOKLINE].ensure((n_tiles + 2) * 8));
    unsigned long long* tile_cnt = ctx->b[B_TOKLINE].as<unsigned long long>();
    CK(cudaMemsetAsync(tile_cnt + n_tiles, 0, 8, s));
    k_tok_count<<<(unsigned)n_tiles, TK_THREADS, 0, s>>>(text, n16, tile_cnt);
    {
        size_t tb = T->cub.cap;
        CK(cub::DeviceScan::ExclusiveSum(T->cub.p, tb, tile_cnt, tile_cnt, (int64_t)(n_tiles + 1), s));
    }
    CK(cudaMemcpyAsync(T->h_tot, tile_cnt + n_tiles, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    const uint64_t n_lines = T->h_tot[0] + (unterminated ? 1 : 0);
    if (n_lines == 0 || n_lines >= 0xFFFFFFF0ull) return PP_TOK_HOST;
    TRY_ALLOC(lines.ensure((n_lines + 2) * 8));
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~size_t(255); return o; };
    const size_t o_rec = carve(n_lines * sizeof(tok::FLineRec)), o_al = carve((n_lines + 1) * 8), o_ns = carve(n_lines * 4), o_rs = carve(n_lines * 4);
    TRY_ALLOC(tmp.ensure(off));
    uint8_t* b = tmp.as<uint8_t>();
    fd->text = text; fd->n = n; fd->n_lines = n_lines; fd->unterminated = unterminated ? 1 : 0;
    fd->line_start = lines.as<unsigned long long>();
    fd->recs = (tok::FLineRec*)(b + o_rec); fd->s_al = (unsigned long long*)(b + o_al);
    fd->name_slot = (uint32_t*)(b + o_ns); fd->ref_slot = (uint32_t*)(b + o_rs);
    k_tok_index<<<(unsigned)n_tiles, TK_THREADS, 0, s>>>(text, n16, tile_cnt, lines.as<unsigned long long>());
    k_ftok_parse<<<(unsigned)((n_lines + 1 + TK_LINE_THREADS - 1) / TK_LINE_THREADS), TK_LINE_THREADS, 0, s>>>(*fd, which, d_st);
    CK(cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, fd->s_al, fd->s_al, (int64_t)(n_lines + 1)));
    CK(T->cub.ensure(cub_bytes + 256));
    {
        size_t tb = T->cub.cap;
        CK(cub::DeviceScan::ExclusiveSum(T->cub.p, tb, fd->s_al, fd->s_al, (int64_t)(n_lines + 1), s));
    }
    *launches += 7;
    return PP_OK;
}

struct TokFilterBufs {                 // device buffers of the filter text path, kept in the tokeniser state
    DevBuf lines[2], tmp[2], mate[2], table, out, status, passkeep;
};

static void free_filter_bufs(TokFilterBufs* b) {
    for (int k = 0; k < 2; ++k) { b->lines[k].release(); b->tmp[k].release(); b->mate[k].release(); }
    b->table.release(); b->out.release(); b->status.release(); b->passkeep.release();
    delete b;
}

// The filter's verdict as the polish records' ZP flag (alignment.rs:72-74): alignment i of the file failed -> PP_FLAG_ZPFAIL.
__global__ void __launch_bounds__(256) k_apply_pass(uint8_t* __restrict__ flags, const uint8_t* __restrict__ pass, uint64_t n) {
    const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
    if (i < n && !pass[i]) flags[i] |= PP_FLAG_ZPFAIL;
}

// `polypolish filter` with the SAM text handled on the device.  PP_OK, PP_TOK_HOST (the host path must do it) or an error
// (the filter's own: no usable pairs, ambiguous orientation; I/O; CUDA).  out1 / out2 may be null (no filtered SAM is written).
// With `fuse`: the two texts, still resident, are then tokenised for `polish` (pp_tok_*) with the filter's verdict taking the
// place of the ZP:Z:fail tag the reference would have written and re-read (filter.rs:334-342, alignment.rs:72-74): the resident
// dataset is what `polish` would load from the filtered files.  fuse->rc = PP_OK / PP_TOK_HOST for that second part.
int pp_filter_files_device(pp_ctx* ctx, const char* in1, const char* in2, const char* out1, const char* out2, const pp_filter_params* prm_in,
                           pp_filter_result* res, pp_filter_file_stats* fs, pp_fused_polish* fuse) {
    CK(cudaSetDevice(ctx->device));
    TokState* T = nullptr;
    int rc = tok_state(ctx, &T);
    if (rc) return rc;
    if (!T->fbufs) T->fbufs = new TokFilterBufs();
    TokFilterBufs& B = *T->fbufs;
    cudaStream_t s = ctx->stream;
    const char* ins[2] = {in1, in2};
    const char* outs[2] = {out1, out2};
    memset(fs, 0, sizeof *fs);
    const auto t_begin = std::chrono::steady_clock::now();
    auto t_mark = t_begin;
    auto lap = [&](int i) { const auto now = std::chrono::steady_clock::now(); fs->phase_ms[i] += std::chrono::duration<float, std::milli>(now - t_mark).count(); t_mark = now; };

    CK(B.status.ensure(sizeof(FStatus)));
    FStatus* d_st = B.status.as<FStatus>();
    FStatus h_st;
    h_st.first_bad[0] = h_st.first_bad[1] = ~0ull; h_st.collision = 0; h_st.pad = 0;
    CK(cudaMemcpyAsync(d_st, &h_st, sizeof h_st, cudaMemcpyHostToDevice, s));
    CK(cudaStreamSynchronize(s));

    // ---- both texts into HBM; the second streams in while the first is indexed and parsed
    FileDev fd[2];
    uint32_t launches = 0;
    float h2d_ms = 0;
    if (T->pf.active && (T->pf.path != in1 || T->pf.strip)) { if (T->pf.th.joinable()) T->pf.th.join(); T->pf.active = false; }
    for (int k = 0; k < 2; ++k) {
        rc = prefetch_wait(ctx, T, ins[k], false);
        if (rc != PP_OK) return rc;
        const int buf = T->pf.buf;
        const uint64_t n = T->pf.n;
        const bool unterminated = n > 0 && T->pf.last != '\n';
        h2d_ms += T->pf.ms;
        fs->text_bytes[k] = n;
        if (k == 0) {
            rc = prefetch_start(ctx, T, ins[1], false);
            if (rc != PP_OK) return rc;
        }
        rc = ftok_lines(ctx, T, k, T->text[buf].as<uint8_t>(), n, unterminated, B.lines[k], B.tmp[k], d_st, &fd[k], &launches);
        if (rc != PP_OK) {
            if (T->pf.active) { if (T->pf.th.joinable()) T->pf.th.join(); T->pf.active = false; }
            return rc;
        }
    }
    CK(cudaMemcpyAsync(T->h_tot + 0, fd[0].s_al + fd[0].n_lines, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(T->h_tot + 1, fd[1].s_al + fd[1].n_lines, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(&h_st, d_st, sizeof h_st, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    const uint64_t n_al[2] = {T->h_tot[0], T->h_tot[1]};
    fs->alignments[0] = n_al[0]; fs->alignments[1] = n_al[1];
    if (h_st.first_bad[0] != ~0ull || h_st.first_bad[1] != ~0ull) return PP_TOK_HOST;
    if (n_al[0] == 0 || n_al[1] == 0) return PP_TOK_HOST;               // "no alignments found in ..." is worded by the host path
    if (n_al[0] >= 0x7FFFFFFFull || n_al[1] >= 0x7FFFFFFFull) return PP_TOK_HOST;
    lap(0);

    // ---- intern QNAMEs and RNAMEs
    uint64_t cap = 1024;
    while (cap < 3 * (n_al[0] + n_al[1]) + 1024) cap <<= 1;
    if (cap > (1ull << 31)) return PP_TOK_HOST;
    TRY_ALLOC(B.table.ensure(cap * 16));
    InternTable tb;
    tb.key = B.table.as<unsigned long long>(); tb.rep = tb.key + cap; tb.mask = (uint32_t)(cap - 1);
    CK(cudaMemsetAsync(tb.key, 0, cap * 8, s));
    CK(cudaMemsetAsync(tb.rep, 0xFF, cap * 8, s));
    for (int k = 0; k < 2; ++k)
        k_ftok_intern<<<(unsigned)((fd[k].n_lines + TK_LINE_THREADS - 1) / TK_LINE_THREADS), TK_LINE_THREADS, 0, s>>>(fd[k], k, tb, d_st);
    Mate mates[2];
    for (int k = 0; k < 2; ++k) {
        k_ftok_verify<<<(unsigned)((fd[k].n_lines + TK_LINE_THREADS - 1) / TK_LINE_THREADS), TK_LINE_THREADS, 0, s>>>(fd[0], fd[1], k, tb, d_st);
        const size_t na = (size_t)n_al[k];
        TRY_ALLOC(B.mate[k].ensure(na * 17 + 5 * 256));
        uint8_t* mb = B.mate[k].as<uint8_t>();
        auto up = [](size_t v) { return (v + 255) & ~size_t(255); };
        MateOut mo;
        mo.name_id = (uint32_t*)mb; mo.contig = (uint32_t*)(mb + up(na * 4)); mo.ref_start = (uint32_t*)(mb + 2 * up(na * 4));
        mo.ref_end = (uint32_t*)(mb + 3 * up(na * 4)); mo.flags = mb + 4 * up(na * 4);
        k_ftok_emit<<<(unsigned)((fd[k].n_lines + TK_LINE_THREADS - 1) / TK_LINE_THREADS), TK_LINE_THREADS, 0, s>>>(fd[k], mo);
        mates[k].name_id = mo.name_id; mates[k].contig = mo.contig; mates[k].ref_start = mo.ref_start; mates[k].ref_end = mo.ref_end;
        mates[k].flags = mo.flags; mates[k].cnt = nullptr; mates[k].head = nullptr; mates[k].next = nullptr; mates[k].pass = nullptr;
        mates[k].n = (uint32_t)na;
    }
    launches += 6;
    CK(cudaMemcpyAsync(&h_st, d_st, sizeof h_st, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    CK(cudaGetLastError());
    if (h_st.collision) return PP_TOK_HOST;
    lap(1);

    // ---- the filter proper (filter_kernels.cu), flags stay on the device
    pp_filter_params prm = *prm_in;
    prm.n_names = cap;
    res->pass1 = nullptr; res->pass2 = nullptr;
    const uint8_t* d_pass[2] = {nullptr, nullptr};
    uint64_t np[2] = {0, 0};
    CK(cudaEventRecord(ctx->ev[0], s));
    rc = pp_filter_core(ctx, mates, &prm, res, d_pass, np);
    if (rc != PP_OK) return rc;
    launches += res->timing.launches;
    lap(2);

    // ---- output text, file by file: lengths -> offsets -> bytes -> the output file
    float d2h_ms = 0;
    for (int k = 0; k < 2; ++k) {
        fs->pass[k] = np[k];
        fs->fail[k] = n_al[k] - np[k];
        if (!outs[k]) continue;
        const uint64_t nl = fd[k].n_lines;
        DevBuf& offs = B.table;                                                 // the intern table is done with: reuse it
        CK(offs.ensure((nl + 2) * 8));
        unsigned long long* out_off = offs.as<unsigned long long>();
        k_ftok_outlen<<<(unsigned)((nl + 1 + TK_LINE_THREADS - 1) / TK_LINE_THREADS), TK_LINE_THREADS, 0, s>>>(fd[k], d_pass[k], out_off);
        size_t cub_bytes = 0;
        CK(cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, out_off, out_off, (int64_t)(nl + 1)));
        CK(T->cub.ensure(cub_bytes + 256));
        {
            size_t tbb = T->cub.cap;
            CK(cub::DeviceScan::ExclusiveSum(T->cub.p, tbb, out_off, out_off, (int64_t)(nl + 1), s));
        }
        CK(cudaMemcpyAsync(T->h_tot, out_off + nl, 8, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        const uint64_t out_n = T->h_tot[0];
        lap(3);
        TRY_ALLOC(B.out.ensure(out_n + 64));
        k_ftok_copy<<<(unsigned)((nl * 32 + 255) / 256), 256, 0, s>>>(fd[k], d_pass[k], out_off, B.out.as<uint8_t>());
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        launches += 4;
        lap(4);
        // A regular file gets its final size up front and is filled in parallel (shared mapping / pwrite at offsets).  Anything
        // else - a FIFO, >(gzip ...), /dev/stdout into a pipe, /dev/null - cannot be truncated or written at offsets: it is
        // streamed in order with write(), like the reference's BufWriter (filter.rs:296-349).
        struct stat osb;
        const bool special = stat(outs[k], &osb) == 0 && !S_ISREG(osb.st_mode);
        const int ofd = special ? open(outs[k], O_WRONLY) : open(outs[k], O_RDWR | O_CREAT | O_TRUNC, 0666);
        if (ofd < 0) return ctx->fail(PP_ERR_IO, std::string("unable to write alignments to \"") + outs[k] + "\"");
        const auto t0 = std::chrono::steady_clock::now();
        int cuda_err = 0;
        int wrc = PP_OK;
        bool stream_out = special;
        if (out_n && !stream_out && ftruncate(ofd, (off_t)out_n) != 0) stream_out = true;
        if (out_n && stream_out) {
            wrc = download_stream(ctx->device, T, B.out.as<uint8_t>(), ofd, out_n, &cuda_err);
        } else if (out_n) {
            // Stores into a mapping cannot report "no space left" (they raise SIGBUS), so the mapping is only used when the
            // file system has room to spare; otherwise pwrite() reports the error like the reference does (filter.rs:307-311).
            struct statvfs vfs;
            const bool roomy = fstatvfs(ofd, &vfs) == 0 && (uint64_t)vfs.f_bavail * (uint64_t)vfs.f_frsize > 2 * out_n + (64ull << 20);
            void* map = roomy ? mmap(nullptr, (size_t)out_n, PROT_READ | PROT_WRITE, MAP_SHARED, ofd, 0) : MAP_FAILED;
            if (map == MAP_FAILED) map = nullptr;
            wrc = download_file(ctx->device, T, B.out.as<uint8_t>(), ofd, (uint8_t*)map, out_n, &cuda_err);
            if (map && munmap(map, (size_t)out_n) != 0 && wrc == PP_OK) wrc = PP_ERR_IO;
        }
        if (close(ofd) != 0 && wrc == PP_OK) wrc = PP_ERR_IO;
        d2h_ms += std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (wrc == PP_ERR_IO) return ctx->fail(PP_ERR_IO, std::string("unable to write alignments to \"") + outs[k] + "\"");
        if (wrc == PP_ERR_CUDA) return ctx->fail_cuda((cudaError_t)cuda_err, "filtered SAM download", __FILE__, __LINE__);
        lap(5);
        fs->out_bytes[k] = out_n;
    }
    fs->h2d_ms = h2d_ms;
    fs->d2h_ms = d2h_ms;
    fs->launches = launches;
    if (fuse) {
        // the verdicts move out of the context's scratch buffer (the tokeniser uses it), then both texts are tokenised in place
        CK(B.passkeep.ensure(n_al[0] + n_al[1] + 64));
        uint8_t* keep = B.passkeep.as<uint8_t>();
        CK(cudaMemcpyAsync(keep, d_pass[0], n_al[0], cudaMemcpyDeviceToDevice, s));
        CK(cudaMemcpyAsync(keep + n_al[0], d_pass[1], n_al[1], cudaMemcpyDeviceToDevice, s));
        CK(cudaStreamSynchronize(s));
        fuse->rc = PP_TOK_HOST;
        int bits = 4;
        for (int attempt = 0; attempt < 2; ++attempt) {
            rc = pp_tok_begin(ctx, fuse->fasta, fuse->careful, bits);
            if (rc != PP_OK) return rc;
            T->expect_total = fd[0].n + fd[1].n;
            memset(fuse->stats, 0, sizeof fuse->stats);
            for (int k = 0; k < 2 && rc == PP_OK; ++k) {
                rc = tok_process(ctx, T, fd[k].text, fd[k].n, fd[k].unterminated != 0, &fuse->stats[k]);
                if (rc == PP_OK && fuse->stats[k].alignments != n_al[k]) rc = PP_TOK_HOST;      // (cannot happen: same lines, same rule)
            }
            if (rc == PP_TOK_NEED8 && bits == 4) { bits = 8; continue; }
            if (rc == PP_TOK_NEED8) rc = PP_TOK_HOST;
            if (rc < 0) return rc;
            if (rc == PP_OK) {
                const uint64_t n = n_al[0] + n_al[1];
                k_apply_pass<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(ctx->b[B_FLAGS].as<uint8_t>(), keep, n);
                CK(cudaStreamSynchronize(s));
                CK(cudaGetLastError());
                rc = pp_tok_finish(ctx);
                if (rc < 0) return rc;
                fuse->n_aln = n;
            }
            fuse->rc = rc;
            break;
        }
    }
    fs->total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    return PP_OK;
}
