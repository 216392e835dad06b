"""The polish kernels themselves (k_prep -> stable sort -> k_bin_bounds -> k_tile -> k_compact, polypolish_b200/csrc/polish_dev.cuh)
run on the CPU through tests/emu (one OS thread per CUDA thread) against the oracle, byte for byte.  This is a logic check of
the device code for runs without a GPU; the real parity tests are the `-m gpu` ones.  PP_EMU_ALL=1 runs every fuzz seed.  The fallback
and boundary paths (long reads, queue overflow, global-k, node-pool and output overflow, long alleles, many contigs) are
tests/test_emu_polish_limits.py, and on the device tests/test_gpu_polish_limits.py."""
import os

import pytest

import polypolish_b200 as pp
from polypolish_b200 import api
from tests import emu_lib, fuzzgen

ALL = bool(os.environ.get("PP_EMU_ALL"))


def check(oracle, fa, sams, grid_tiles=2, **opts):
    try:
        exp = ("ok", oracle.polish(fa, sams, **opts))
    except Exception as e:
        exp = ("err", e.msg)
    f = pp.load_fasta(fa)
    try:
        p = pp.pack_sams(f, sams, careful=opts.get("careful", False))
    except pp.PolypolishError as e:
        assert exp[0] == "err"                      # a text-level error: the packer's business, not the kernels'
        return None
    r = emu_lib.polish(f, p, grid_tiles=grid_tiles, **opts)
    if exp[0] == "err":
        assert "error" in r, exp[1]
        assert r["error"].split()[0] in exp[1]
        return r
    assert "error" not in r, r
    assert emu_lib.fasta_bytes(f, r["sequences"]) == exp[1]["fasta"]
    assert r["changed"] == exp[1]["changed"] and r["zero_depth"] == exp[1]["zero_depth"] and r["n_aln_used"] == exp[1]["used_total"]
    for got, want in zip(r["total_depth"], exp[1]["total_depth"]):
        assert abs(got - want) <= 1e-9 * max(1.0, abs(want))
    return r


@pytest.mark.parametrize("seed", list(range(100, 180)) if ALL else [100, 101, 104, 107, 112, 116, 121, 133, 140, 152, 164, 175])
def test_emu_fuzz(oracle, tmp_path, seed):
    case = fuzzgen.make_case(seed, exotic=0.5 if seed % 4 == 0 else 0.0)
    fa, sams = case.write(tmp_path)
    check(oracle, fa, sams, **case.opts)


@pytest.mark.parametrize("seed", list(range(300, 312)) if ALL else [300, 303, 307])
def test_emu_fuzz_deep_multimap(oracle, tmp_path, seed):
    """Most reads multi-mapped: non-dyadic k everywhere -> the ordered depth walk (merge of the bins by alignment index)."""
    case = fuzzgen.make_case(seed, n_contigs=2, contig_len=(200, 400), depth=(150, 300), multimap=0.8, opts=dict(careful=False))
    fa, sams = case.write(tmp_path)
    check(oracle, fa, sams, **case.opts)


def test_emu_synth_tiles(oracle, tmp_path):
    """Several tiles, several CTAs sharing them by ticket, reads that straddle tile and bin borders, repeats (k = 7, 5, 3)."""
    syn = api.Synth(seed=21, n_contigs=2, contig_len=9_000, depth=40)
    fa, sams = syn.write(tmp_path)
    check(oracle, fa, sams, grid_tiles=3)
    check(oracle, fa, sams, grid_tiles=1, careful=True)


@pytest.mark.parametrize("seed", [400, 401, 402, 403] if ALL else [400, 402])
def test_emu_long_reads(oracle, tmp_path, seed):
    """Reads of 200-900 bases over several tiles: more than 256 entries (a tile looks two bins back), more than 512 (the
    long list every tile scans), longer than the 192-base register path, indels next to tile borders."""
    case = fuzzgen.make_case(seed, n_contigs=2, contig_len=(2500, 5000), depth=(15, 30), read_len=(200, 900), multimap=0.4,
                             opts=dict(careful=False))
    fa, sams = case.write(tmp_path)
    check(oracle, fa, sams, grid_tiles=2, **case.opts)


def test_emu_hand_made_edges(oracle, tmp_path):
    """Homopolymer tails of 32+ bases (the fast path hands over to the general walk), reads that are one base, reads trimmed to
    nothing, both strands, reads ending exactly on a contig end and on a tile border (position 2048)."""
    import random
    rng = random.Random(7)
    ctg = "".join(rng.choice("ACGT") for _ in range(2000)) + "A" * 60 + "".join(rng.choice("ACGT") for _ in range(1500)) + "C" * 45
    fa = tmp_path / "e.fasta"
    fa.write_text(">edge\n" + ctg + "\n")

    def rc(s):
        return s[::-1].translate(str.maketrans("ACGT", "TGCA"))
    lines = []
    n = 0

    def add(pos0, length, reverse=False, dup=1):
        nonlocal n
        seq = ctg[pos0:pos0 + length]
        for _ in range(dup):
            # SEQ is always given on the forward reference strand in SAM; flag 16 only marks the strand
            lines.append(f"r{n}\t{16 if reverse else 0}\tedge\t{pos0 + 1}\t60\t{length}M\t*\t0\t0\t{seq}\t*\tNM:i:0")
            n += 1
    for rev in (False, True):
        add(1950, 100, rev, 6)        # ends inside the A run: tail of 50 A (> 32)
        add(1990, 70, rev, 6)         # entirely a homopolymer tail after 10 bases
        add(2000, 60, rev, 3)         # all one base: trimmed to nothing
        add(1900, 148, rev, 6)        # crosses the tile border at 2048
        add(2047, 1, rev, 2)          # one base
        add(3400, len(ctg) - 3400, rev, 6)   # to the contig end (C run of 45)
        add(len(ctg) - 40, 40, rev, 3)
        add(1000, 192, rev, 5)        # longest fast-path read
        add(1000, 193, rev, 5)        # first general-path read
    # secondaries without SEQ taking the reverse complement of the source
    lines.append(f"m0\t0\tedge\t101\t60\t80M\t*\t0\t0\t{ctg[100:180]}\t*\tNM:i:0")
    lines.append(f"m0\t272\tedge\t501\t0\t80M\t*\t0\t0\t*\t*\tNM:i:3")
    lines.append(f"m0\t256\tedge\t901\t0\t80M\t*\t0\t0\t*\t*\tNM:i:3")
    sam = tmp_path / "e.sam"
    sam.write_text("\n".join(lines) + "\n")
    check(oracle, fa, [sam], grid_tiles=2, min_depth=2)
    check(oracle, fa, [sam], grid_tiles=1, min_depth=0, fraction_invalid=0.05)
