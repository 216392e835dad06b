"""BAM input without a GPU: the host reader and the records' SAM text (bam.cpp, through the host packer), the device decoder's
per-record bodies (bam_rec.h, through tests/bam_harness.cpp), and pp_synth_write_bam.

The BAM writer below is plain Python (struct + zlib), written from SAMv1 §4; a hand-assembled known-answer file guards against the
writer and the reader sharing one misreading."""
import ctypes as C
import gzip
import os
import struct
import subprocess
import tempfile
import zlib

import numpy as np
import pytest

from tests import fuzzgen
import polypolish_b200 as pp
from polypolish_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
PP_OK, PP_TOK_HOST, PP_TOK_NEED8 = 0, 1, 2
CODES = "=ACMGRSVTWYHKDBN"
OPS = "MIDNSHP=X"
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


# ---- writing BAM -------------------------------------------------------------------------------------------------------------
def bgzf(data, block=65280, cuts=None):
    """BGZF of `data`: blocks of `block` bytes (or cut at the offsets in `cuts`), then the end-of-file block."""
    bounds = sorted(set([0, len(data)] + list(cuts or []))) if cuts is not None else list(range(0, len(data), block)) + [len(data)]
    out = bytearray()
    for a, b in zip(bounds, bounds[1:]):
        chunk = data[a:b]
        c = zlib.compressobj(6, zlib.DEFLATED, -15)
        cd = c.compress(chunk) + c.flush()
        out += struct.pack("<BBBBIBBHBBHH", 31, 139, 8, 4, 0, 0, 255, 6, 66, 67, 2, len(cd) + 25)
        out += cd + struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk))
    return bytes(out) + BGZF_EOF


def int_tag(tag, v, typ=None):
    if typ is None:
        typ = "C" if 0 <= v <= 255 else "c" if -128 <= v < 0 else "S" if 0 <= v <= 65535 else "s" if -32768 <= v < 0 else "I" if v >= 0 else "i"
    fmt = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I"}[typ]
    return tag.encode() + typ.encode() + struct.pack("<" + fmt, v)


def record(qname, flag, ref, pos, mapq, cigar_ops, seq, aux=b"", next_ref=-1, next_pos=-1, tlen=0, qual=None):
    """One BAM record: cigar_ops = [(len, op code)], seq = bases (str), pos 0-based."""
    name = qname.encode("latin-1") + b"\0"
    cig = b"".join(struct.pack("<I", (n << 4) | o) for n, o in cigar_ops)
    s = seq.upper()
    packed = bytes(((CODES.index(s[i]) << 4) | (CODES.index(s[i + 1]) if i + 1 < len(s) else 0)) for i in range(0, len(s), 2))
    q = bytes([0xFF] * len(s)) if qual is None else bytes(qual)
    body = struct.pack("<iiBBHHHIiii", ref, pos, len(name), mapq, 4680, len(cigar_ops), flag, len(s), next_ref, next_pos, tlen)
    body += name + cig + packed + q + aux
    return struct.pack("<I", len(body)) + body


def header(text, refs):
    t = text.encode("latin-1")
    out = b"BAM\1" + struct.pack("<I", len(t)) + t + struct.pack("<I", len(refs))
    for name, ln in refs:
        n = name.encode("latin-1") + b"\0"
        out += struct.pack("<I", len(n)) + n + struct.pack("<I", ln)
    return out


def parse_cigar(c):
    if c == "*":
        return []
    out, num = [], ""
    for ch in c:
        if ch.isdigit():
            num += ch
        else:
            out.append((int(num), OPS.index(ch)))
            num = ""
    return out


def sam_to_bam_stream(text, nm_type=None):
    """The uncompressed BAM stream of a SAM text (header lines -> header text; empty lines dropped).  Tags: NM/AS/XS -> integer
    types (nm_type forces NM's), Z tags as Z."""
    lines = [ln[:-1] if ln.endswith("\r") else ln for ln in text.split("\n")]
    htext = "".join(ln + "\n" for ln in lines if ln.startswith("@"))
    refs = []
    for ln in lines:
        if ln.startswith("@SQ"):
            f = dict(x.split(":", 1) for x in ln.split("\t")[1:] if ":" in x)
            refs.append((f["SN"], int(f.get("LN", 0))))
    names = [r[0] for r in refs]
    recs = []
    for ln in lines:
        if not ln or ln.startswith("@"):
            continue
        f = ln.split("\t")
        for r in (f[2], f[6]):
            if r not in ("*", "=") and r not in names:
                names.append(r)
                refs.append((r, 1000))
        ref = -1 if f[2] == "*" else names.index(f[2])
        nref = -1 if f[6] == "*" else ref if f[6] == "=" else names.index(f[6])
        aux = b""
        for t in f[11:]:
            tag, typ, val = t.split(":", 2)
            if typ == "i":
                aux += int_tag(tag, int(val), nm_type if tag == "NM" else None)
            else:
                aux += tag.encode() + b"Z" + val.encode("latin-1") + b"\0"
        seq = "" if f[9] == "*" else f[9]
        recs.append(record(f[0], int(f[1]), ref, int(f[3]) - 1, int(f[4]), parse_cigar(f[5]), seq, aux, nref, int(f[7]) - 1, int(f[8])))
    return header(htext, refs), recs


def write_bam(path, hdr, recs, block=65280, span=False):
    """span: cut the BGZF blocks inside records (every record boundary + 7)."""
    data = hdr + b"".join(recs)
    cuts = None
    if span:
        cuts, at = [], len(hdr)
        for r in recs:
            cuts.append(at + min(7, len(r) - 1))
            at += len(r)
    with open(path, "wb") as fh:
        fh.write(bgzf(data, block, cuts))
    return path


def sam_file_to_bam(sam_path, bam_path, **kw):
    nm_type = kw.pop("nm_type", None)
    hdr, recs = sam_to_bam_stream(open(sam_path, encoding="latin-1").read(), nm_type)
    return write_bam(bam_path, hdr, recs, **kw)


# ---- helpers ------------------------------------------------------------------------------------------------------------------
def pack(fasta_path, files, careful=False):
    f = pp.load_fasta(fasta_path)
    p = api.Packed(f, careful)
    for x in files:
        p.add_file(x)
    p.finish()
    return f, p


def assert_same(a, b):
    for k, v in b.items():
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, a[k]), k
        else:
            assert v == a[k], k


def same_arrays(fasta_path, sams, bams, careful=False):
    _, ps = pack(fasta_path, sams, careful)
    _, pb = pack(fasta_path, bams, careful)
    assert_same(pb.arrays(), ps.arrays())
    for i in range(ps.arrays()["contig"].size):
        assert pb.read_name(i) == ps.read_name(i)
    return ps


def pack_error(fasta_path, files):
    with pytest.raises(api.PolypolishError) as e:
        pack(fasta_path, files)
    return e.value


# ---- the known-answer file -----------------------------------------------------------------------------------------------------
# Written by hand from SAMv1 §4.2: header "@SQ\tSN:c1\tLN:40\n", one reference "c1" (40 bp), three records:
#   r1  flag 0   c1 pos 2 (0-based 1)  CIGAR 4M     SEQ ACGT  NM:C:1
#   r1  flag 16  c1 pos 9              CIGAR 2S2M   SEQ *     NM:C:0  zp:Z:FAIL
#   u   flag 4   refID -1 pos -1       CIGAR *      SEQ AC    (no tags)
def kat_stream():
    text = b"@SQ\tSN:c1\tLN:40\n"
    h = b"BAM\x01" + bytes.fromhex("10000000") + text + bytes.fromhex("01000000" "03000000") + b"c1\x00" + bytes.fromhex("28000000")
    r1 = bytes.fromhex(
        "00000000"      # refID 0
        "01000000"      # pos 1
        "03" "3c"       # l_read_name 3, mapq 60
        "4812"          # bin 4680
        "0100"          # n_cigar_op 1
        "0000"          # flag 0
        "04000000"      # l_seq 4
        "ffffffff" "ffffffff" "00000000") + b"r1\x00" + bytes.fromhex(
        "40000000"      # 4M
        "1248"          # A C G T = 1 2 4 8
        "ffffffff"      # QUAL missing
        ) + b"NMC\x01"
    r2 = bytes.fromhex(
        "00000000" "08000000" "03" "3c" "4812" "0200" "1000" "00000000" "ffffffff" "ffffffff" "00000000") + b"r1\x00" + bytes.fromhex(
        "24000000"      # 2S
        "20000000"      # 2M
        ) + b"NMC\x00" + b"zpZFAIL\x00"
    r3 = bytes.fromhex(
        "ffffffff" "ffffffff" "02" "00" "4812" "0000" "0400" "02000000" "ffffffff" "ffffffff" "00000000") + b"u\x00" + bytes.fromhex(
        "12" "ffff")
    recs = [struct.pack("<I", len(r)) + r for r in (r1, r2, r3)]
    return h, recs


def test_known_answer_bam(tmp_path):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "A" * 40 + "\n")
    h, recs = kat_stream()
    bam = write_bam(str(tmp_path / "k.bam"), h, recs)
    f, p = pack(str(fa), [bam])
    a = p.arrays()
    assert a["n_reads"] == 1 and a["seq_bits"] == 4
    assert a["contig"].tolist() == [0, 0]
    assert a["ref_start"].tolist() == [1, 8]
    assert a["read_id"].tolist() == [0, 0]
    assert a["nm"].tolist() == [1, 0]
    assert a["n_cigar"].tolist() == [1, 2]
    assert a["cigar_ops"].tolist() == [(4 << 4) | 0, (2 << 4) | 4, (2 << 4) | 0]
    assert a["seq_len"].tolist() == [4, 4]                    # the SEQ=* record takes its group's sequence
    assert a["seq_off"].tolist() == [0, 0]
    assert a["flags"].tolist() == [0, 0x01 | 0x02 | 0x04 | 0x08]   # reverse, ZP fail, SEQ *, reverse complement of the source
    assert a["seq_pool"][:2].tolist() == [0x21, 0x84]         # A C G T, low nibble first
    assert p.read_name(0) == "r1" and p.read_name(1) == "r1"
    # the same as the SAM text of the file
    sam = tmp_path / "k.sam"
    sam.write_text("@SQ\tSN:c1\tLN:40\nr1\t0\tc1\t2\t60\t4M\t*\t0\t0\tACGT\t*\tNM:i:1\n"
                   "r1\t16\tc1\t9\t60\t2S2M\t*\t0\t0\t*\t*\tNM:i:0\tzp:Z:FAIL\nu\t4\t*\t0\t0\t*\t*\t0\t0\tAC\t*\n")
    same_arrays(str(fa), [str(sam)], [bam])


# ---- equality with the SAM text: golden fixtures and fuzz cases ------------------------------------------------------------------
GOLDEN_CASES = sorted(d for d in os.listdir(GOLDEN) if d.startswith("polish_"))


@pytest.mark.parametrize("name", GOLDEN_CASES)
@pytest.mark.parametrize("layout", ["default", "tiny", "span"])
def test_golden_bam_equals_sam(tmp_path, name, layout):
    d = os.path.join(GOLDEN, name)
    sams = sorted(os.path.join(d, x) for x in os.listdir(d) if x.endswith(".sam"))
    kw = dict(default={}, tiny=dict(block=61), span=dict(span=True))[layout]
    bams = [sam_file_to_bam(s, str(tmp_path / (os.path.basename(s) + ".bam")), **kw) for s in sams]
    same_arrays(os.path.join(d, "asm.fasta"), sams, bams, careful=False)


def fuzz_files(tmp_path, seed, exotic=0.0, nm_type=None, **kw):
    case = fuzzgen.make_case(seed, exotic=exotic, multimap=0.5 if seed % 2 else 0.25)
    fa = tmp_path / "a.fasta"
    fa.write_text(case.fasta_text)
    sams, bams = [], []
    for i, t in enumerate(case.sam_texts):
        s = tmp_path / f"r{i}.sam"
        s.write_bytes(t.encode("latin-1"))
        sams.append(str(s))
        bams.append(sam_file_to_bam(str(s), str(tmp_path / f"r{i}.bam"), nm_type=nm_type, **kw))
    return case, str(fa), sams, bams


@pytest.mark.parametrize("seed", range(300, 340))
def test_fuzz_bam_equals_sam(tmp_path, seed):
    nm_type = [None, "c", "S", "I", "i"][seed % 5]
    case, fa, sams, bams = fuzz_files(tmp_path, seed, nm_type=nm_type, block=[65280, 997, 64][seed % 3])
    same_arrays(fa, sams, bams, case.opts["careful"])
    # and mixed with the SAM files, in either order
    _, pt = pack(fa, [sams[0], sams[-1]], case.opts["careful"])
    for mixed in ([sams[0], bams[-1]], [bams[0], sams[-1]]):
        _, pm = pack(fa, mixed, case.opts["careful"])
        assert_same(pm.arrays(), pt.arrays())


def edge_sam():
    L = lambda *f: "\t".join(str(x) for x in f) + "\n"
    return ("@SQ\tSN:c1\tLN:60\n@SQ\tSN:c2\tLN:60\n" +
            L("a", 0, "c1", 3, 60, "5M0I3M", "*", 0, 0, "ACGTRYKMN", "*", "NM:i:2", "ZP:Z:Fail") +          # zero-length op, IUPAC
            L("a", 256, "*", 7, 0, "9M", "*", 0, 0, "*", "*", "NM:i:0") +                                   # refID -1 on an aligned record
            L("a", 4, "*", 0, 0, "*", "*", 0, 0, "ACG", "*") +                                               # unaligned inside the group
            L("a", 272, "c2", 1, 0, "9M", "*", 0, 0, "*", "*", "NM:i:1", "zP:Z:faiL") +
            L("b", 16, "c2", 20, 60, "4M", "*", 0, 0, "TTGA", "*", "NM:i:0", "ZP:Z:failed") +
            L("", 0, "c1", 1, 60, "4M", "*", 0, 0, "ACGT", "*", "NM:i:0") +                                   # empty QNAME joins what follows
            L("c", 0, "c1", 1, 60, "4M", "*", 0, 0, "AC=T", "*", "NM:i:0"))                                   # '=': 8-bit pool


@pytest.mark.parametrize("nm_type", ["c", "C", "s", "S", "i", "I"])
def test_edge_records(tmp_path, nm_type):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n>c2\n" + "TTGA" * 15 + "\n")
    sam = tmp_path / "e.sam"
    sam.write_text(edge_sam())
    hdr, recs = sam_to_bam_stream(edge_sam(), nm_type)
    bam = write_bam(str(tmp_path / "e.bam"), hdr, recs, span=True)
    ps = same_arrays(str(fa), [str(sam)], [bam])
    assert ps.arrays()["seq_bits"] == 8


def test_long_cigar_placeholder(tmp_path):
    """kSmN with a CG:B:I array stands for the CIGAR in CG."""
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n")
    ops = [(2, 0), (1, 1), (3, 0)]
    cg = b"CGBI" + struct.pack("<I", 3) + b"".join(struct.pack("<I", (n << 4) | o) for n, o in ops)
    r = record("r", 0, 0, 4, 60, [(6, 4), (5, 3)], "ACGTAC", int_tag("NM", 1) + cg)
    bam = write_bam(str(tmp_path / "l.bam"), header("", [("c1", 60)]), [r])
    sam = tmp_path / "l.sam"
    sam.write_text("r\t0\tc1\t5\t60\t2M1I3M\t*\t0\t0\tACGTAC\t*\tNM:i:1\n")
    same_arrays(str(fa), [str(sam)], [bam])


# ---- errors -------------------------------------------------------------------------------------------------------------------
def err_case(tmp_path, sam_text):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n")
    sam = tmp_path / "x.sam"
    sam.write_text(sam_text)
    hdr, recs = sam_to_bam_stream(sam_text)
    bam = write_bam(str(tmp_path / "x.bam"), hdr, recs)
    es, eb = pack_error(str(fa), [str(sam)]), pack_error(str(fa), [bam])
    return str(es).replace(str(sam), "F"), str(eb).replace(bam, "F"), es, eb


def test_missing_nm_same_line_number(tmp_path):
    text = "@HD\tVN:1.6\n@SQ\tSN:c1\tLN:60\n@CO\tthree header lines\nr\t0\tc1\t1\t60\t4M\t*\t0\t0\tACGT\t*\tNM:i:0\ns\t0\tc1\t1\t60\t4M\t*\t0\t0\tACGT\t*\n"
    ms, mb, es, eb = err_case(tmp_path, text)
    assert "missing NM tag" in ms and "(line 5)" in ms
    assert ms == mb and es.code == eb.code


def test_invalid_cigar_same_message(tmp_path):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n")
    r = record("r", 0, 0, 0, 60, [(2, 0), (2, 9)], "ACGT", int_tag("NM", 0))      # op 9 is 'B' in SAM text
    bam = write_bam(str(tmp_path / "x.bam"), header("@SQ\tSN:c1\tLN:60\n", [("c1", 60)]), [r])
    sam = tmp_path / "x.sam"
    sam.write_text("@SQ\tSN:c1\tLN:60\nr\t0\tc1\t1\t60\t2M2B\t*\t0\t0\tACGT\t*\tNM:i:0\n")
    es, eb = pack_error(str(fa), [str(sam)]), pack_error(str(fa), [bam])
    assert str(eb) == str(es) and "invalid CIGAR string for read r" in str(eb)


def test_negative_nm_same_message(tmp_path):
    ms, mb, es, eb = err_case(tmp_path, "r\t0\tc1\t1\t60\t4M\t*\t0\t0\tACGT\t*\tNM:i:-3\n")
    assert ms == mb and "invalid NM tag" in ms


def good_bam(tmp_path):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n")
    recs = [record(f"r{i}", 0, 0, i, 60, [(4, 0)], "ACGT", int_tag("NM", 0)) for i in range(40)]
    data = bgzf(header("@SQ\tSN:c1\tLN:60\n", [("c1", 60)]) + b"".join(recs), block=300)
    return str(fa), data


@pytest.mark.parametrize("damage,what", [
    (lambda d: d[:len(d) - 28 - 40], "truncated BGZF block"),
    (lambda d: d[:len(d) - 28], "no BGZF end-of-file block"),
    (lambda d: d[:60] + bytes([d[60] ^ 0x40]) + d[61:], "mismatch"),
    (lambda d: d + b"junk that is not BGZF at all", "not BGZF"),
])
def test_bam_structural_errors(tmp_path, damage, what):
    fa, data = good_bam(tmp_path)
    bam = tmp_path / "d.bam"
    bam.write_bytes(damage(data))
    e = pack_error(fa, [str(bam)])
    assert e.code == api.PP_ERR_IO
    assert str(bam) in str(e) and "not a valid BAM file" in str(e) and what in str(e)


def test_bam_record_faults(tmp_path):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n")
    hdr = header("", [("c1", 60)])
    good = record("r", 0, 0, 0, 60, [(4, 0)], "ACGT", int_tag("NM", 0))
    cases = [
        (record("r", 0, 3, 0, 60, [(4, 0)], "ACGT", int_tag("NM", 0)), "refID or next_refID out of range"),
        (record("r", 0, 0, 0, 60, [(4, 0)], "ACGT", b"NMC"), "malformed optional fields"),
        (good[:-6], "runs past"),
    ]
    for rec, what in cases:
        rec = struct.pack("<I", len(rec) - 4) + rec[4:]
        bam = write_bam(str(tmp_path / "f.bam"), hdr, [good, rec])
        e = pack_error(str(fa), [bam])
        assert e.code == api.PP_ERR_IO and "record 2" in str(e) and what in str(e), str(e)


def test_plain_gzip_and_sam_are_not_bam(tmp_path):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n")
    text = "r\t0\tc1\t1\t60\t4M\t*\t0\t0\tACGT\t*\tNM:i:0\n"
    sam = tmp_path / "x.sam"
    sam.write_text(text)
    pack(str(fa), [str(sam)])
    gz = tmp_path / "x.sam.gz"
    gz.write_bytes(gzip.compress(text.encode()))
    e = pack_error(str(fa), [str(gz)])                 # parsed as SAM text, as before: the gzip bytes are not a SAM line
    assert "BAM" not in str(e)
    # a BGZF file whose content is not BAM (bgzip'ed SAM) is SAM too
    bg = tmp_path / "x.sam.bgz"
    bg.write_bytes(bgzf(text.encode()))
    e2 = pack_error(str(fa), [str(bg)])
    assert "BAM" not in str(e2)
    # a .bam name does not make SAM text BAM
    named = tmp_path / "y.bam"
    named.write_text(text)
    pack(str(fa), [str(named)])


# ---- the device decoder's per-record bodies on the CPU ------------------------------------------------------------------------
@pytest.fixture(scope="module")
def H():
    out = os.path.join(tempfile.mkdtemp(prefix="bam_harness_"), "bam_harness.so")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", out, os.path.join(ROOT, "tests", "bam_harness.cpp")])
    return C.CDLL(out)


def bam_cpu(H, f, streams, careful=False, bits=4):
    total = sum(len(h) + sum(len(r) for r in rs) for h, rs in streams)
    cap_aln, cap_ops, cap_seq = total // 30 + 16, total // 4 + 16, total * 2 + 4096
    a = dict(contig=np.zeros(cap_aln, np.uint32), ref_start=np.zeros(cap_aln, np.uint32), read_id=np.zeros(cap_aln, np.uint32),
             seq_off=np.zeros(cap_aln, np.uint32), seq_len=np.zeros(cap_aln, np.uint16), cigar_off=np.zeros(cap_aln, np.uint32),
             n_cigar=np.zeros(cap_aln, np.uint16), nm=np.zeros(cap_aln, np.uint32), flags=np.zeros(cap_aln, np.uint8),
             cigar_ops=np.zeros(cap_ops, np.uint32), seq_pool=np.full(cap_seq, 0xEE, np.uint8))
    order = ["contig", "ref_start", "read_id", "seq_off", "seq_len", "cigar_off", "n_cigar", "nm", "flags", "cigar_ops", "seq_pool"]
    counts = (C.c_uint64 * 6)()
    H.bam_cpu.restype = C.c_int
    for h, rs in streams:
        data = h + b"".join(rs)
        # refID -> contig, as pp::BamImage builds it: exact name lookup ("*" for refID -1)
        n_ref = struct.unpack_from("<I", h, 8 + struct.unpack_from("<I", h, 4)[0])[0]
        names, p = [], 12 + struct.unpack_from("<I", h, 4)[0]
        for _ in range(n_ref):
            ln = struct.unpack_from("<I", h, p)[0]
            names.append(h[p + 4:p + 4 + ln - 1].decode("latin-1"))
            p += 8 + ln
        rc_tab = (C.c_uint32 * (n_ref + 1))(*[f.names.index(n) if n in f.names else 0xFFFFFFFF for n in ["*"] + names])
        rc = H.bam_cpu(C.c_char_p(data), C.c_uint64(len(data)), rc_tab, C.c_uint32(n_ref), C.c_int(int(careful)), C.c_int(bits),
                       C.c_uint64(cap_aln), C.c_uint64(cap_ops), C.c_uint64(cap_seq), *[a[k].ctypes.data_as(C.c_void_p) for k in order], counts)
        if rc != PP_OK:
            return rc, None
    n, no, nb = counts[0], counts[1], counts[2]
    out = {k: a[k][:n].copy() for k in order[:9]}
    out["cigar_ops"] = a["cigar_ops"][:no].copy()
    out["seq_pool"] = a["seq_pool"][:nb * (16 if bits == 4 else 32)].copy()
    out["n_reads"] = counts[3]
    out["seq_bits"] = bits
    return PP_OK, out


@pytest.mark.parametrize("seed", range(300, 316))
def test_bam_rec_bodies_equal_host_packer(H, tmp_path, seed):
    case = fuzzgen.make_case(seed, exotic=0.0, multimap=0.5 if seed % 2 else 0.25)
    fa = tmp_path / "a.fasta"
    fa.write_text(case.fasta_text)
    streams = [sam_to_bam_stream(t, ["c", "C", "s", "S", "i", "I"][seed % 6]) for t in case.sam_texts]
    bams = [write_bam(str(tmp_path / f"r{i}.bam"), h, rs) for i, (h, rs) in enumerate(streams)]
    f, p = pack(str(fa), bams, case.opts["careful"])
    host = p.arrays()
    rc, dev = bam_cpu(H, f, streams, case.opts["careful"], int(host["seq_bits"]))
    assert rc == PP_OK
    assert_same(dev, host)


def test_bam_rec_bodies_edge_records(H, tmp_path):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n>c2\n" + "TTGA" * 15 + "\n")
    f, p = pack(str(fa), [write_bam(str(tmp_path / "e.bam"), *sam_to_bam_stream(edge_sam()))])
    s = sam_to_bam_stream(edge_sam())
    assert bam_cpu(H, f, [s], bits=4)[0] == PP_TOK_NEED8
    rc, dev = bam_cpu(H, f, [s], bits=8)
    assert rc == PP_OK
    assert_same(dev, p.arrays())


def test_bam_rec_bodies_leave_wording_to_the_host(H, tmp_path):
    fa = tmp_path / "a.fasta"
    fa.write_text(">c1\n" + "ACGT" * 15 + "\n")
    f = pp.load_fasta(str(fa))
    hdr = header("", [("c1", 60)])
    ok = record("r", 0, 0, 0, 60, [(4, 0)], "ACGT", int_tag("NM", 0))
    for bad in [record("r", 0, 0, 0, 60, [(4, 10)], "ACGT", int_tag("NM", 0)),             # op code above 8
                record("r", 0, 0, 0, 60, [(4, 0)], "ACGT", int_tag("NM", -2, "c")),         # negative NM
                record("r", 0, 0, 0, 60, [(4, 0)], "ACGT"),                                  # missing NM
                record("r", 0, 0, 0, 60, [(4, 4), (9, 3)], "ACGT", int_tag("NM", 0)),       # kSmN
                record("@r", 0, 0, 0, 60, [(4, 0)], "ACGT", int_tag("NM", 0)),              # a header line in SAM
                record("r", 0, 0, 0, 60, [(4, 0)], "ACGT", int_tag("NM", 0) + b"ZPZfa\til\0"),
                record("r", 0, 0, -2, 60, [(4, 0)], "ACGT", int_tag("NM", 0))]:             # POS -1: "invalid POS field"
        assert bam_cpu(H, f, [(hdr, [ok, bad])])[0] == PP_TOK_HOST
    assert bam_cpu(H, f, [(hdr, [ok, ok])])[0] == PP_OK


# ---- synthetic BAM ------------------------------------------------------------------------------------------------------------
def test_synth_write_bam_equals_write_sam(tmp_path):
    syn = api.Synth(seed=5, contig_len=20_000, depth=20, n_contigs=2)
    os.makedirs(tmp_path / "s")
    os.makedirs(tmp_path / "b")
    fa, sams = syn.write(tmp_path / "s")
    fb, bams = syn.write(tmp_path / "b", bam=True)
    assert all(open(b, "rb").read(4) == b"\x1f\x8b\x08\x04" for b in bams)
    assert all(open(b, "rb").read()[-28:] == BGZF_EOF for b in bams)
    same_arrays(fa, sams, bams)
