// emu_polish.cpp — runs the polish kernels of polypolish_b200/csrc/polish_dev.cuh on the CPU (tests/emu/cuda_emu.h): the same
// device code, one OS thread per CUDA thread, so that the kernels' logic is checked against the oracle without a GPU.
// TEST INFRASTRUCTURE: built and used by tests/test_emu_polish.py only; nothing in polypolish_b200/ links or loads this.
#include "cuda_emu.h"

#include "../../polypolish_b200/csrc/polish_dev.cuh"

#include <numeric>
#include <string>

namespace {

void init_comp_table() {
    for (int i = 0; i < 256; ++i) c_comp[i] = 'N';
    const char* a = "ATGCNRYSWKMBVDH.-?";
    const char* b = "TACGNYRSWMKVBHD.-?";
    for (int i = 0; a[i]; ++i) c_comp[(unsigned char)a[i]] = (uint8_t)b[i];
}

// What one emulated call saw, for tests that check a fallback path was taken (the device keeps the same numbers in DevStatus).
struct EmuReport {
    int first_rc;                    // return code of the first pass (100: FL_BIGGROUP, the global-k pass followed)
    unsigned flags;                  // DevStatus.flags of the last pass
    unsigned node_count;             // other-allele nodes the last pass asked for (may exceed node_cap)
    unsigned global_k;               // the last pass ran k_classify_multi + goodk<true>
    unsigned long long out_len;      // polished bases of the last pass
    unsigned long long node_cap, out_cap;   // capacities the last pass ran with
    int guards_ok;                   // the words right after the node pool and the output buffer are untouched
};

constexpr uint32_t GUARD32 = 0xA5C3F00Du;
constexpr size_t GUARD_NODES = 4, GUARD_OUT = 64;

template <int BITS>
int run(const pp_contigs* c, const pp_alignments* a, const pp_polish_params* prm, pp_polish_result* res, int grid_tiles, bool global_k,
        uint64_t node_cap_req, uint64_t out_cap_req, EmuReport* rep, uint64_t* err_out) {
    const uint64_t G = c->off[c->n_contigs], n_aln = a->n_aln;
    const uint32_t n_tiles = (uint32_t)((G + TL_T - 1) / TL_T), n_bins = (uint32_t)((G + PP_BIN - 1) >> PP_BIN_SHIFT);
    const size_t padG = (size_t)n_tiles * TL_T + 16;
    std::vector<uint8_t> draft(padG + 4096, 0);
    memcpy(draft.data(), c->bases, G);
    std::vector<uint8_t> seq_pool(a->seq_pool_bytes + 512, 0);
    if (a->seq_pool_bytes) memcpy(seq_pool.data(), a->seq_pool, a->seq_pool_bytes);
    // 16-byte aligned copies (uint4 loads)
    std::vector<uint4> draft16((draft.size() + 15) / 16), pool16((seq_pool.size() + 15) / 16);
    memcpy(draft16.data(), draft.data(), draft.size());
    memcpy(pool16.data(), seq_pool.data(), seq_pool.size());
    std::vector<uint32_t> cigar_ops(a->n_cigar_ops + 16, 0);
    if (a->n_cigar_ops) memcpy(cigar_ops.data(), a->cigar_ops, a->n_cigar_ops * 4);

    std::vector<TileRec> recs(n_aln + 16), srec(n_aln + 16);
    std::vector<uint32_t> key(n_aln + 16), val(n_aln + 16), skey(n_aln + 16), sval(n_aln + 16), bin_start(n_bins + 4, 0), kf(n_aln + 16, 0xDEADBEEFu);
    std::vector<uint4> wrec(n_aln + 16, make_uint4(0xDEADBEEFu, 0xDEADBEEFu, 0xDEADBEEFu, 0xDEADBEEFu));
    std::vector<uint4> sseq((n_aln + 16) * TL_SEQ_QUADS + 16, make_uint4(0xCDCDCDCDu, 0xCDCDCDCDu, 0xCDCDCDCDu, 0xCDCDCDCDu));
    std::vector<uint8_t> errc(n_aln + 16, 0xEE);
    std::vector<uint16_t> gq(n_aln + 16, 0xEEEE);
    std::vector<uint32_t> oth_head(((size_t)(G + TL_T - 1) / TL_T) * TL_T + 16, 0xEEEEEEEEu), kcount(a->n_reads + 2, 0);   // (k_tile zeroes the heads itself)
    // node pool and output buffer: today's sizes unless the caller asks for others, each followed by guard words
    const uint64_t node_cap = node_cap_req ? node_cap_req : std::max<uint64_t>(1 << 16, n_aln * 4 + G);
    std::vector<OthNode> nodes(node_cap + GUARD_NODES);
    for (size_t i = node_cap; i < nodes.size(); ++i) { nodes[i].sig = nodes[i].val = 0xA5C3F00DA5C3F00Dull; nodes[i].count = nodes[i].next = GUARD32; }
    std::vector<unsigned long long> changed(c->n_contigs, 0), zero(c->n_contigs, 0), out_off(c->n_contigs + 1, 0);
    std::vector<double> tdepth(c->n_contigs, 0.0);
    std::vector<uint16_t> resv(padG, 0);
    std::vector<uint32_t> rec_at(G + 1, 0);
    std::vector<long long> chunk_delta(n_tiles, 0);
    const uint64_t out_cap = out_cap_req ? out_cap_req : G + G / 4 + (1u << 20);
    std::vector<uint8_t> out(out_cap + GUARD_OUT);
    memset(out.data() + out_cap, 0xA5, GUARD_OUT);
    DevStatus st;
    memset(&st, 0, sizeof st);
    st.err = ~0ull;
    DevParams dp{prm->fraction_valid, prm->fraction_invalid, prm->min_depth, prm->max_errors, prm->careful ? 1 : 0, 0};

    DevData d;
    memset(&d, 0, sizeof d);
    d.n_aln = n_aln;
    d.contig = a->contig; d.ref_start = a->ref_start; d.read_id = a->read_id; d.seq_off = a->seq_off; d.cigar_off = a->cigar_off; d.nm = a->nm;
    d.cigar_ops = cigar_ops.data(); d.seq_len = a->seq_len; d.n_cigar = a->n_cigar; d.flags = a->flags;
    d.seq_pool = (const uint8_t*)pool16.data(); d.draft = (const uint8_t*)draft16.data();
    d.contig_off = (const unsigned long long*)c->off; d.n_contigs = c->n_contigs; d.G = (uint32_t)G; d.n_bins = n_bins; d.n_tiles = n_tiles;
    d.k = kcount.data(); d.recs = recs.data(); d.key = key.data(); d.val = val.data(); d.sval = sval.data(); d.bin_start = bin_start.data();
    d.srec = srec.data(); d.sseq = sseq.data(); d.kf = kf.data(); d.errc = errc.data(); d.gq = gq.data();
    d.wrec = wrec.data(); d.oth_head = oth_head.data(); d.nodes = nodes.data(); d.node_cap = (uint32_t)node_cap; d.prm = &dp; d.st = &st;
    VoteParams vp;
    vp.n_chunks = n_tiles; vp.out = out.data(); vp.out_cap = out_cap; vp.out_off = out_off.data(); vp.changed = changed.data();
    vp.zero_depth = zero.data(); vp.total_depth = tdepth.data(); vp.res = resv.data(); vp.rec_at = rec_at.data(); vp.chunk_delta = chunk_delta.data();
    vp.dbg = nullptr;

    // ---- once per dataset: bin, stable sort, bounds, permute
    if (n_aln) {
        emu::launch(3, 256, 0, [&] { bin_body<BITS>(d); });
        std::vector<uint32_t> order(n_aln);
        std::iota(order.begin(), order.end(), 0u);
        std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return key[x] < key[y]; });   // = the stable radix sort
        for (uint64_t i = 0; i < n_aln; ++i) { skey[i] = key[order[i]]; sval[i] = val[order[i]]; }
    }
    emu::launch((unsigned)((n_aln + 1 + 255) / 256), 256, 0, [&] { bin_bounds_body(skey.data(), (uint32_t)n_aln, n_bins + 2, bin_start.data()); });
    d.n_slots = bin_start[n_bins + 1];
    d.max_ext = st.max_ext;
    if (d.n_slots) {
        emu::launch((d.n_slots + 255) / 256, 256, 0, [&] { permute_body(d); });
        if (BITS == 4) emu::launch((unsigned)(((uint64_t)d.n_slots * TL_SEQ_QUADS + 255) / 256), 256, 0, [&] { permute_seq_body(d); });
    }
    std::vector<uint32_t> tweight(n_tiles + 1), tindex(n_tiles + 1), torder(n_tiles + 1);
    emu::launch((n_tiles + 255) / 256, 256, 0, [&] { tile_weight_body(d, tweight.data(), tindex.data()); });
    {
        std::vector<uint32_t> o(n_tiles);
        std::iota(o.begin(), o.end(), 0u);
        std::stable_sort(o.begin(), o.end(), [&](uint32_t x, uint32_t y) { return tweight[x] > tweight[y]; });
        for (uint32_t i = 0; i < n_tiles; ++i) torder[i] = tindex[o[i]];
    }
    d.tile_order = torder.data();
    // ---- per call
    if (n_aln && global_k) emu::launch(2, 256, 0, [&] { k_classify_multi(d); });
    if (n_aln)
        emu::launch(2, PR_THREADS, sizeof(PrepShared), [&] {
            PrepShared& sh = *(PrepShared*)emu::shared_base();
            if (global_k) goodk_body<true>(d, sh); else goodk_body<false>(d, sh);
        });
    emu::launch((unsigned)std::max(1, std::min<int>(grid_tiles, (int)n_tiles)), TL_THREADS, sizeof(TileShared), [&] {
        tile_body<BITS>(d, vp, *(TileShared*)emu::shared_base());
    });
    emu::launch(n_tiles, VT_THREADS, sizeof(CompactShared), [&] { compact_body<BITS>(d, vp, *(CompactShared*)emu::shared_base()); });

    *err_out = st.err;
    bool guards = true;
    for (size_t i = node_cap; i < nodes.size(); ++i)
        guards = guards && nodes[i].sig == 0xA5C3F00DA5C3F00Dull && nodes[i].val == 0xA5C3F00DA5C3F00Dull && nodes[i].count == GUARD32 &&
                 nodes[i].next == GUARD32;
    for (size_t i = out_cap; i < out.size(); ++i) guards = guards && out[i] == 0xA5;
    rep->flags = st.flags; rep->node_count = st.node_count; rep->global_k = global_k ? 1 : 0; rep->out_len = st.out_len;
    rep->node_cap = node_cap; rep->out_cap = out_cap; rep->guards_ok = guards ? 1 : 0;
    res->out_len = st.out_len;
    res->n_aln_used = st.n_used;
    res->error_aln = st.err == ~0ull ? -1 : (int64_t)(st.err >> 8);
    if (st.err != ~0ull) return PP_ERR_INPUT;
    if (st.flags & FL_BIGGROUP) return 100;
    if (st.flags & (FL_NODE_OVF | FL_OUT_OVF)) return PP_ERR_NOMEM;
    if (res->out_bases) {
        if (res->out_cap < st.out_len) return PP_ERR_ARG;
        memcpy(res->out_bases, out.data(), st.out_len);
        if (res->out_off) memcpy(res->out_off, out_off.data(), (c->n_contigs + 1) * 8);
        if (res->changed) memcpy(res->changed, changed.data(), c->n_contigs * 8);
        if (res->zero_depth) memcpy(res->zero_depth, zero.data(), c->n_contigs * 8);
        if (res->total_depth) memcpy(res->total_depth, tdepth.data(), c->n_contigs * 8);
    }
    return PP_OK;
}

}  // namespace

// The polish kernels on the CPU.  grid_tiles = CTAs of k_tile (they share tiles through the ticket, like on the device).
// node_cap / out_cap: capacity of the other-allele node pool and of the output buffer, 0 = the default sizes (node_cap max(65536,
// 4 n_aln + G), out_cap G + G/4 + 1 MiB).  Unlike the device, the emulator does not grow them and repeat: an overflow is returned as
// PP_ERR_NOMEM.  rep (may be null) receives what the call saw.
extern "C" int emu_polish_ex(const pp_contigs* c, const pp_alignments* a, const pp_polish_params* prm, pp_polish_result* res, int grid_tiles,
                             unsigned long long node_cap, unsigned long long out_cap, EmuReport* rep, unsigned long long* err_code) {
    init_comp_table();
    uint64_t err = 0;
    EmuReport local;
    if (!rep) rep = &local;
    memset(rep, 0, sizeof *rep);
    auto pass = [&](bool global_k) {
        return a->seq_bits == 4 ? run<4>(c, a, prm, res, grid_tiles, global_k, node_cap, out_cap, rep, &err)
                                : run<8>(c, a, prm, res, grid_tiles, global_k, node_cap, out_cap, rep, &err);
    };
    int rc = pass(false);
    rep->first_rc = rc;
    if (rc == 100) rc = pass(true);
    if (err_code) *err_code = err;
    return rc;
}

// The same with the default capacities and no report (the original entry point; its signature stays as it was).
extern "C" int emu_polish(const pp_contigs* c, const pp_alignments* a, const pp_polish_params* prm, pp_polish_result* res, int grid_tiles,
                          unsigned long long* err_code) {
    return emu_polish_ex(c, a, prm, res, grid_tiles, 0, 0, nullptr, err_code);
}

// The allele signature helpers of polish_dev.cuh on their own (tests/test_emu_polish_limits.py compares them with plain string
// comparison).  An allele = `len` symbols from `start` of the effective read (reverse-complemented if rc) at block offset off_blk.
extern "C" unsigned long long emu_make_sig(int bits, const uint8_t* pool, uint32_t off_blk, uint32_t slen, int rc, uint32_t start, uint32_t len) {
    init_comp_table();
    return bits == 4 ? make_sig<4>(pool, off_blk, slen, rc != 0, start, len) : make_sig<8>(pool, off_blk, slen, rc != 0, start, len);
}
extern "C" int emu_sig_exact(int bits, unsigned long long sig) { return bits == 4 ? sig_exact<4>(sig) : sig_exact<8>(sig); }
extern "C" int emu_allele_equal(int bits, const uint8_t* pool, uint32_t off_a, uint32_t slen_a, int rc_a, uint32_t start_a, uint32_t len_a,
                                uint32_t off_b, uint32_t slen_b, int rc_b, uint32_t start_b, uint32_t len_b) {
    init_comp_table();
    const uint32_t seq_off[2] = {off_a, off_b};
    const uint16_t seq_len[2] = {(uint16_t)slen_a, (uint16_t)slen_b};
    const uint8_t flags[2] = {(uint8_t)(rc_a ? PP_FLAG_RC : 0), (uint8_t)(rc_b ? PP_FLAG_RC : 0)};
    const SeqRef r{pool, seq_off, seq_len, flags};
    const unsigned long long va = (0ull << 32) | ((unsigned long long)start_a << 16) | len_a, vb = (1ull << 32) | ((unsigned long long)start_b << 16) | len_b;
    return bits == 4 ? allele_equal<4>(r, va, vb) : allele_equal<8>(r, va, vb);
}
