"""BAM input on the GPU: the device decoder (tok_kernels.cu k_bam_parse / k_bam_emit) against the host packer, and `polish` of BAM
files against the oracle's `polish` of their SAM text - FASTA, log numbers, --debug TSV, errors, several contexts, full size."""
import os
import shutil
import tempfile

import pytest

import polypolish_b200 as pp
from polypolish_b200 import api
from tests import fuzzgen
from tests.test_bam_cpu import (GOLDEN, GOLDEN_CASES, assert_same, edge_sam, pack, record, header, int_tag, sam_file_to_bam,
                                sam_to_bam_stream, write_bam)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import __graft_entry__ as g
    g.build()
    c = pp.Context(0)
    yield c
    c.close()


def golden(name, tmp_path, **kw):
    d = os.path.join(GOLDEN, name)
    sams = sorted(os.path.join(d, x) for x in os.listdir(d) if x.endswith(".sam"))
    bams = [sam_file_to_bam(s, str(tmp_path / (os.path.basename(s)[:-4] + ".bam")), **kw) for s in sams]
    import json
    opts = json.load(open(os.path.join(d, "opts.json")))
    return os.path.join(d, "asm.fasta"), sams, bams, opts


def fuzz(tmp_path, seed, **kw):
    case = fuzzgen.make_case(seed, exotic=0.0, multimap=0.5 if seed % 2 else 0.25)
    fa = tmp_path / "a.fasta"
    fa.write_text(case.fasta_text)
    sams, bams = [], []
    for i, t in enumerate(case.sam_texts):
        s = tmp_path / f"r{i}.sam"
        s.write_bytes(t.encode("latin-1"))
        sams.append(str(s))
        bams.append(sam_file_to_bam(str(s), str(tmp_path / f"r{i}.bam"), nm_type=["c", "S", "I", None][seed % 4], **kw))
    return str(fa), sams, bams, case.opts


def log_lines(text, names):
    """stderr of a verbose run without its timing lines, file names replaced by their index."""
    out = []
    for ln in text.splitlines():
        if ln.startswith(("SAM tokeniser", "BAM decoder", "GPU job", "read groups exchanged")):
            continue
        for i, n in enumerate(names):
            ln = ln.replace(n, f"<{i}>")
        out.append(ln)
    return out


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_device_arrays_from_bam(ctx, tmp_path, name):
    fa, sams, bams, opts = golden(name, tmp_path, block=500)
    f, p = pack(fa, sams, opts["careful"])
    rc, st = ctx.tokenise(f, bams, careful=opts["careful"], seq_bits=4)
    assert rc == 0
    assert st[0]["lines"] > 0
    assert_same(ctx.dataset_arrays(), p.arrays())


def test_device_arrays_from_bam_eight_bit(ctx, tmp_path):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n>c2\n" + "TTGA" * 15 + "\n")
    sam = tmp_path / "e.sam"
    sam.write_text(edge_sam())
    bam = write_bam(str(tmp_path / "e.bam"), *sam_to_bam_stream(edge_sam()), span=True)
    f, p = pack(str(fa), [str(sam)])
    assert p.arrays()["seq_bits"] == 8
    rc, _ = ctx.tokenise(f, [bam], seq_bits=4)
    assert rc == 2                                          # PP_TOK_NEED8
    rc, _ = ctx.tokenise(f, [bam], seq_bits=8)
    assert rc == 0
    assert_same(ctx.dataset_arrays(), p.arrays())


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_polish_bam_golden_equals_oracle(ctx, tmp_path, name, capfd):
    fa, sams, bams, opts = golden(name, tmp_path)
    d = os.path.join(GOLDEN, name)
    ctx.set_parser(0)
    capfd.readouterr()
    got = ctx.polish_files(fa, sams, verbose=True, **opts)
    log_sam = log_lines(capfd.readouterr().err, sams)
    got_b = ctx.polish_files(fa, bams, debug=str(tmp_path / "dbg.tsv"), **opts)
    assert got_b == open(os.path.join(d, "expected.fasta"), "rb").read() == got
    assert open(tmp_path / "dbg.tsv", "rb").read() == open(os.path.join(d, "expected_debug.tsv"), "rb").read()
    capfd.readouterr()
    ctx.polish_files(fa, bams, verbose=True, **opts)
    assert log_lines(capfd.readouterr().err, bams) == log_sam


@pytest.mark.parametrize("seed", range(400, 412))
def test_polish_bam_fuzz_equals_oracle(ctx, oracle, tmp_path, seed):
    fa, sams, bams, opts = fuzz(tmp_path, seed, block=[65280, 777, 90][seed % 3])
    o = {k: opts[k] for k in ("careful", "fraction_invalid", "fraction_valid", "max_errors", "min_depth") if k in opts}
    try:
        exp = oracle.polish(fa, sams, debug=True, **o)
    except Exception as e:                                  # the oracle's error: the BAM run must end with the same message
        with pytest.raises(api.PolypolishError) as ge:
            ctx.polish_files(fa, bams, **o)
        assert str(e).split("] ")[-1] in str(ge.value)
        return
    ctx.set_parser(0)
    assert ctx.polish_files(fa, bams, debug=str(tmp_path / "d.tsv"), **o) == exp["fasta"]
    assert open(tmp_path / "d.tsv", "rb").read() == exp["debug_tsv"]
    assert ctx.polish_files(fa, bams, **o) == exp["fasta"]
    # SAM and BAM mixed, in both orders
    if len(sams) > 1:
        assert ctx.polish_files(fa, [sams[0], bams[1]] + bams[2:], **o) == exp["fasta"]
        assert ctx.polish_files(fa, [bams[0], sams[1]] + sams[2:], **o) == exp["fasta"]


def test_errors_match_host_parse(ctx, tmp_path):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n")
    ok = record("r", 0, 0, 0, 60, [(4, 0)], "ACGT", int_tag("NM", 0))
    hdr = header("@SQ\tSN:c1\tLN:60\n@CO\tx\n", [("c1", 60)])
    cases = [record("s", 0, 0, 0, 60, [(4, 0)], "ACGT"),                          # missing NM tag (line 4)
             record("s", 0, 0, 0, 60, [(4, 0), (2, 9)], "ACGT", int_tag("NM", 0)), # invalid CIGAR
             record("s", 0, 0, 0, 60, [(4, 0)], "ACGT", int_tag("NM", -1, "c")),    # invalid NM tag
             record("s", 0, 1, 0, 60, [(4, 0)], "ACGT", int_tag("NM", 0))]          # refID out of range
    first = None
    for i, bad in enumerate(cases):
        bam = write_bam(str(tmp_path / f"e{i}.bam"), hdr, [ok, bad])
        msgs = []
        for parser in (0, 1):
            ctx.set_parser(parser)
            with pytest.raises(api.PolypolishError) as e:
                ctx.polish_files(str(fa), [bam])
            msgs.append((e.value.code, e.value.msg))
        ctx.set_parser(0)
        assert msgs[0] == msgs[1], msgs
        first = first or msgs[0][1]
    assert "missing NM tag" in first and "(line 4)" in first


@pytest.mark.parametrize("seed", [401, 403, 405, 407])
def test_multi_context_bam_equals_one(ctx, tmp_path, seed):
    """3 contexts on one GPU: each decodes its record range of the one image, cut between read groups."""
    fa, sams, bams, opts = fuzz(tmp_path, seed)
    o = {k: opts[k] for k in ("careful", "fraction_invalid", "fraction_valid", "max_errors", "min_depth") if k in opts}
    try:
        one = ctx.polish_files(fa, bams, **o)
    except api.PolypolishError:
        return
    ctxs = [pp.Context(0) for _ in range(3)]
    try:
        assert api.polish_files_multi(fa, bams, contexts=ctxs, **o) == one
        assert api.polish_files_multi(fa, [sams[0]] + bams[1:], contexts=ctxs, **o) == one
    finally:
        for c in ctxs:
            c.close()


def test_multi_context_cuts_inside_groups_with_unaligned(ctx, tmp_path):
    """Groups whose unaligned records and empty names sit where the equal-count cuts fall."""
    fa = tmp_path / "a.fasta"
    seq = "ACGTTGCA" * 40
    fa.write_text(">c1\n" + seq + "\n>c2\n" + seq[::-1] + "\n>c3\n" + seq[3:] + seq[:3] + "\n")
    lines = ["@SQ\tSN:c1\tLN:320", "@SQ\tSN:c2\tLN:320", "@SQ\tSN:c3\tLN:320"]
    for g in range(30):
        name = "" if g % 7 == 3 else f"g{g}"
        for k in range(4):
            if k == 2:
                lines.append(f"{name}\t4\t*\t0\t0\t*\t*\t0\t0\tACGT\t*")
            else:
                c = (g + k) % 3 + 1
                ref = [seq, seq[::-1], seq[3:] + seq[:3]][c - 1]
                pos = (g * 7 + k * 11) % 280
                s = ref[pos:pos + 30] if k == 0 else "*"
                lines.append(f"{name}\t{0 if k == 0 else 256}\tc{c}\t{pos + 1}\t60\t30M\t*\t0\t0\t{s}\t*\tNM:i:0")
    text = "\n".join(lines) + "\n"
    sam = tmp_path / "g.sam"
    sam.write_text(text)
    bam = write_bam(str(tmp_path / "g.bam"), *sam_to_bam_stream(text), block=100)
    one = ctx.polish_files(str(fa), [str(sam)], min_depth=1)
    ctxs = [pp.Context(0) for _ in range(3)]
    try:
        assert api.polish_files_multi(str(fa), [bam], contexts=ctxs, min_depth=1) == one
    finally:
        for c in ctxs:
            c.close()


def test_config2_full_size_bam(ctx):
    """BASELINE config 2 (5 Mbp x 100x) written as BAM: the FASTA of the SAM run."""
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > (5 << 30) else None
    d = tempfile.mkdtemp(prefix="pp_bam_", dir=base)
    try:
        syn = api.Synth(seed=2, contig_len=5_000_000, depth=100)
        fa, sams = syn.write(d)
        os.makedirs(os.path.join(d, "b"))
        _, bams = syn.write(os.path.join(d, "b"), bam=True)
        ctx.set_parser(0)
        exp = ctx.polish_files(fa, sams)
        assert ctx.polish_files(fa, bams) == exp
        # ... and the records went through the device decoder, not the host packer
        rc, st = ctx.tokenise(pp.load_fasta(fa), bams)
        assert rc == 0 and all(s["alignments"] > 0 and s["device_ms"] > 0 for s in st)
    finally:
        shutil.rmtree(d, ignore_errors=True)
