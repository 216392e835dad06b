"""The polish kernels' fallback and boundary paths on the device, against the CPU oracle, byte for byte (cases: tests/limitcases.py,
at the size that crosses each device threshold): long reads and the long list, one-indel reads at the edges of the two-segment
fast walk, a queue overflow in the 4-bit and the 8-bit pool, read groups too large for k_goodk's scan (global-k, with and without
the memset reset), thousands of short contigs, a node-pool overflow, an output-buffer overflow.  Every case also asserts that
its threshold was crossed, so that a change of a constant cannot turn it into a no-op:
  polish_dev.cuh: TL_FAST_LEN 192, TL_LONG_E 512, PP_BIN 256 (look-back), TL_QCAP 1024, SC_GROUP_SCAN_LIMIT 8192, CP_STAGE 4096;
  polish_kernels.cu:280-281: first node pool max(65,536, n_aln/8 + G/64), first output buffer G + G/16 + 1 MiB;
  polish_kernels.cu:405: the per-call reset block travels as one copy up to PP_INIT_IMAGE (64 KiB), else memsets."""
import pytest

import polypolish_b200 as pp
from polypolish_b200 import api
from tests import fuzzgen, limitcases as lc
from tests.emu_lib import fasta_bytes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import __graft_entry__ as g
    g.build()
    c = pp.Context(0)
    yield c
    c.close()


CASES = {
    "long_reads": lambda: lc.long_reads("gpu"),
    "one_indel_bounds": lambda: lc.one_indel_bounds("gpu"),
    "queue_overflow_4bit": lambda: lc.queue_overflow("gpu", seq_bits=4),
    "queue_overflow_8bit": lambda: lc.queue_overflow("gpu", seq_bits=8),
    "big_group_9000": lambda: lc.big_group("gpu", n_records=9_000),
    "big_group_20000": lambda: lc.big_group("gpu", n_records=20_000),
    "big_group_many_reads": lambda: lc.big_group("gpu", n_records=9_000, many_reads=True),
    "many_contigs": lambda: lc.many_contigs("gpu"),
    "other_allele_flood": lambda: lc.other_allele_flood("gpu"),
    "long_insertions_4bit": lambda: lc.long_insertions("gpu", seq_bits=4),
    "long_insertions_8bit": lambda: lc.long_insertions("gpu", seq_bits=8),
}


def assert_path_ran(name, info, p, r):
    """The threshold quantity of the case against the formula it must cross; r = the polish_packed result."""
    G = info.get("G")
    if name.startswith("big_group"):
        assert info["group_size"] > lc.SC_GROUP_SCAN_LIMIT + lc.PR_THREADS and info["group_start"] % lc.PR_THREADS != 0
        assert r["timing"]["launches"] == 4                   # k_classify_multi + k_goodk<true> + k_tile + k_compact
        if name.endswith("many_reads"):
            assert info["reset_bytes"] > lc.PP_INIT_IMAGE
        return
    assert r["timing"]["launches"] == 3
    if name == "long_reads":
        assert 2 * lc.PP_BIN >= info["max_binned_E"] > lc.PP_BIN and info["n_long"] > 0
        assert info["max_len"] == lc.MAX_U16 and 3 in info["k"]
    elif name == "one_indel_bounds":
        assert 0 < info["n_fast1"] < info["n_one_indel"]
    elif name.startswith("queue_overflow"):
        assert info["deferred_in_tile0"] > lc.TL_QCAP + 100
        assert p.view.seq_bits == (8 if name.endswith("8bit") else 4)
    elif name == "many_contigs":
        assert info["reset_bytes"] > lc.PP_INIT_IMAGE and info["max_contigs_in_8"] > 1
    elif name == "other_allele_flood":
        assert info["distinct_other"] > lc.first_node_cap(p.view.n_aln, G)
    elif name.startswith("long_insertions"):
        assert info["max_chunk_bytes"] > lc.CP_STAGE
        assert r["out_len"] > lc.first_out_cap(G) and r["out_len"] > G + (1 << 20)   # device repeat, then the caller's retry
        assert p.view.seq_bits == (8 if name.endswith("8bit") else 4)


@pytest.mark.parametrize("name", list(CASES))
def test_limit_parity(ctx, oracle, tmp_path, name):
    """FASTA through the file path, the --debug TSV, the statistics through the packed path, and the proof the path ran."""
    case, info = CASES[name]()
    fa, sams = case.write(tmp_path)
    exp = oracle.polish(fa, sams, debug=True, **case.opts)
    assert ctx.polish_files(fa, sams, **case.opts) == exp["fasta"]
    dbg = tmp_path / "debug.tsv"
    assert ctx.polish_files(fa, sams, debug=dbg, **case.opts) == exp["fasta"]
    assert dbg.read_bytes() == exp["debug_tsv"]
    f = pp.load_fasta(fa)
    p = pp.pack_sams(f, sams, careful=case.opts["careful"])
    r = ctx.polish_packed(f.view, p.view, **case.opts)
    assert fasta_bytes(f, r["sequences"]) == exp["fasta"]
    assert r["changed"] == exp["changed"] and r["zero_depth"] == exp["zero_depth"] and r["n_aln_used"] == exp["used_total"]
    for got, want in zip(r["total_depth"], exp["total_depth"]):
        assert abs(got - want) <= 1e-9 * max(1.0, abs(want))
    assert_path_ran(name, info, p, r)


@pytest.mark.parametrize("name", ["big_group_9000", "other_allele_flood", "long_insertions_4bit"])
def test_resident_state_across_calls(ctx, oracle, tmp_path, name):
    """The global-k switch and the grown node pool / output buffer stay with the resident dataset across calls with other options,
    and a new upload starts from the first guesses again."""
    case, info = CASES[name]()
    fa, sams = case.write(tmp_path)
    f = pp.load_fasta(fa)
    p = pp.pack_sams(f, sams)
    ctx.upload(f.view, p.view)
    for opts in (dict(), dict(careful=True), dict(max_errors=2)):
        o = dict(case.opts, **opts)
        r = ctx.polish_resident(**o)
        assert fasta_bytes(f, r["sequences"]) == oracle.polish(fa, sams, **o)["fasta"], opts
    small = fuzzgen.make_case(101)
    d = tmp_path / "small"
    d.mkdir()
    fa2, sams2 = small.write(d)
    f2 = pp.load_fasta(fa2)
    p2 = pp.pack_sams(f2, sams2, careful=small.opts["careful"])
    ctx.upload(f2.view, p2.view)
    r = ctx.polish_resident(**small.opts)
    assert fasta_bytes(f2, r["sequences"]) == oracle.polish(fa2, sams2, **small.opts)["fasta"]
    assert r["timing"]["launches"] == 3


@pytest.mark.parametrize("n", [2, 3])
def test_big_group_several_contexts(oracle, tmp_path, n):
    """pp_polish_files_multi with a read group larger than a context's byte range (ranges are cut only where a group ends, so one
    can be empty)."""
    case, info = lc.big_group("gpu", n_records=20_000)
    fa, sams = case.write(tmp_path)
    exp = oracle.polish(fa, sams, **case.opts)["fasta"]
    ctxs = [pp.Context(0) for _ in range(n)]
    try:
        assert api.polish_files_multi(fa, sams, contexts=ctxs, **case.opts) == exp
    finally:
        for c in ctxs:
            c.close()
