"""The polish kernels' fallback and boundary paths (tests/limitcases.py) run on the CPU through tests/emu against the oracle, byte for
byte: long reads and the long list, one-indel reads at the edges of the two-segment fast walk, a tile whose queue overflows, a read
group too large for k_goodk's scan (global-k), thousands of short contigs, a flood of other alleles, long insertions around the
exact-signature limit and past k_compact's stage.  The node pool and the output buffer are also run too small (the emulator
reports the overflow the device would repeat on, and the words right behind them stay untouched), then at the size the device's
grow rule picks.  The allele signature helpers are checked against plain string comparison.  The same cases at device size are
tests/test_gpu_polish_limits.py.  PP_EMU_ALL=1 also runs the larger variants."""
import ctypes as C
import os
import random

import pytest

import polypolish_b200 as pp
from tests import emu_lib, limitcases as lc
from tests.test_emu_polish import check

ALL = bool(os.environ.get("PP_EMU_ALL"))


def run(oracle, tmp_path, case, grid_tiles=2, **extra):
    fa, sams = case.write(tmp_path)
    r = check(oracle, fa, sams, grid_tiles=grid_tiles, **dict(case.opts, **extra))
    assert r is not None and "error" not in r
    return r


def packed(tmp_path, case):
    fa, sams = case.write(tmp_path)
    f = pp.load_fasta(fa)
    return fa, sams, f, pp.pack_sams(f, sams, careful=case.opts["careful"])


def test_long_reads(oracle, tmp_path):
    case, info = lc.long_reads("gpu" if ALL else "emu")
    # binned reads of up to 512 entries: a tile looks two bins back (3 bins + the long list in the ordered depth walk); longer ones
    # sit in the long list; reads longer than the fast path; the 16-bit read length at its limit; non-dyadic k over all of them
    assert 2 * lc.PP_BIN >= info["max_binned_E"] > lc.PP_BIN
    assert info["n_long"] > 0 and info["max_len"] == lc.MAX_U16 and 3 in info["k"]
    run(oracle, tmp_path, case, grid_tiles=3)
    if ALL:
        run(oracle, tmp_path, case, grid_tiles=1, min_depth=2, fraction_invalid=0.1)


def test_one_indel_bounds(oracle, tmp_path):
    case, info = lc.one_indel_bounds()
    assert 0 < info["n_fast1"] < info["n_one_indel"]          # both sides of every TR_FAST1 edge
    _, _, _, p = packed(tmp_path, case)
    assert p.view.seq_bits == 4                                # (TR_FAST1 is a 4-bit-pool path)
    run(oracle, tmp_path, case)
    run(oracle, tmp_path, case, min_depth=3, fraction_valid=0.6)


@pytest.mark.parametrize("seq_bits", [4, 8])
def test_queue_overflow(oracle, tmp_path, seq_bits):
    case, info = lc.queue_overflow(seq_bits=seq_bits)
    assert info["deferred_in_tile0"] > lc.TL_QCAP + 100
    _, _, _, p = packed(tmp_path, case)
    assert p.view.seq_bits == seq_bits
    run(oracle, tmp_path, case, grid_tiles=1)


@pytest.mark.parametrize("n_records,many_reads", [(9_000, False)] + ([(20_000, False), (9_000, True)] if ALL else []))
def test_big_group(oracle, tmp_path, n_records, many_reads):
    case, info = lc.big_group(n_records=n_records, many_reads=many_reads)
    assert info["group_size"] > lc.SC_GROUP_SCAN_LIMIT + lc.PR_THREADS and info["group_start"] % lc.PR_THREADS != 0
    assert info["good"]["default"] != info["good"]["max_errors=2"]          # k depends on the options
    for opts in (dict(), dict(max_errors=2), dict(careful=True)):
        o = dict(case.opts, **opts)
        fa, sams = case.write(tmp_path)
        r = check(oracle, fa, sams, **o)
        if o["careful"]:                   # --careful drops every multi-record group before k is needed: no scan, no fallback
            assert r["report"]["first_rc"] == 0 and r["report"]["global_k"] == 0, r["report"]
        else:
            assert r["report"]["first_rc"] == emu_lib.BIGGROUP_RC and r["report"]["global_k"] == 1, r["report"]


def test_many_contigs(oracle, tmp_path):
    case, info = lc.many_contigs()
    assert info["max_contigs_in_8"] > 1 and info["n_short"] > 100
    r = run(oracle, tmp_path, case)
    exp = oracle.polish(*case.write(tmp_path), **case.opts)
    assert sum(1 for c in exp["changed"] if c) > len(exp["changed"]) // 2 and sum(exp["zero_depth"]) > 0
    assert r["changed"] == exp["changed"]
    run(oracle, tmp_path, case, min_depth=0)


def test_other_allele_flood_and_node_pool(oracle, tmp_path):
    case, info = lc.other_allele_flood("gpu" if ALL else "emu")
    assert info["distinct_other"] > 10_000
    fa, sams, f, p = packed(tmp_path, case)
    exp = oracle.polish(fa, sams, **case.opts)
    # a pool smaller than the distinct alleles: FL_NODE_OVF, nothing written past the pool
    small = info["distinct_other"] // 3
    r = emu_lib.polish(f, p, node_cap=small, **case.opts)
    assert "overflow" in r and r["overflow"]["flags"] & emu_lib.FL_NODE_OVF, r
    assert r["overflow"]["guards_ok"] == 1 and r["overflow"]["node_count"] > small
    # the device's grow rule (polish_kernels.cu:487) from what the failed call counted, then parity
    n = r["overflow"]["node_count"]
    r = emu_lib.polish(f, p, node_cap=n + n // 4 + 1024, **case.opts)
    assert "overflow" not in r and r["report"]["guards_ok"] == 1 and r["report"]["flags"] == 0
    assert r["report"]["node_count"] >= info["distinct_other"]
    assert emu_lib.fasta_bytes(f, r["sequences"]) == exp["fasta"]
    assert r["changed"] == exp["changed"] and r["n_aln_used"] == exp["used_total"]
    run(oracle, tmp_path, case)


@pytest.mark.parametrize("seq_bits", [4, 8])
def test_long_insertions_and_output_buffer(oracle, tmp_path, seq_bits):
    case, info = lc.long_insertions(seq_bits=seq_bits)
    assert info["max_chunk_bytes"] > lc.CP_STAGE                # one chunk compacted without the shared-memory stage
    fa, sams, f, p = packed(tmp_path, case)
    assert p.view.seq_bits == seq_bits
    exp = oracle.polish(fa, sams, **case.opts)
    out_len = len(b"".join(exp["fasta"].split(b"\n")[1::2]))
    assert out_len >= info["G"] + info["voted_in"] - 16
    # an output buffer smaller than the result: FL_OUT_OVF, nothing written past it
    r = emu_lib.polish(f, p, out_cap=out_len // 2, **case.opts)
    assert "overflow" in r and r["overflow"]["flags"] & emu_lib.FL_OUT_OVF, r
    assert r["overflow"]["guards_ok"] == 1 and r["overflow"]["out_len"] == out_len
    # the device's repeat size (polish_kernels.cu:488), then parity; and exactly the output's size
    for cap in (out_len + 64, out_len):
        r = emu_lib.polish(f, p, out_cap=cap, **case.opts)
        assert "overflow" not in r and r["report"]["guards_ok"] == 1
        assert emu_lib.fasta_bytes(f, r["sequences"]) == exp["fasta"]
    r = run(oracle, tmp_path, case)
    run(oracle, tmp_path, case, fraction_invalid=0.4, fraction_valid=0.6)


# ---- the allele signature helpers of polish_dev.cuh against plain string comparison ---------------------------------------------
NIB = {c: i for i, c in enumerate("=ACMGRSVTWYHKDBN")}


def pool_bytes(seqs, bits):
    """One PP_SEQ_BLOCK-aligned block run per sequence, as the packer lays them out: (pool, block offsets)."""
    block = 32
    out, offs = bytearray(), []
    for s in seqs:
        offs.append(len(out) // (16 if bits == 4 else 32))
        if bits == 4:
            b = bytearray((len(s) + 1) // 2)
            for i, ch in enumerate(s):
                b[i >> 1] |= NIB[ch] << ((i & 1) * 4)
        else:
            b = bytearray(s.encode())
        b += bytes(-len(b) % (block // 2 if bits == 4 else block))
        out += b
    return bytes(out) + bytes(64), offs


@pytest.mark.parametrize("bits", [4, 8])
def test_allele_signatures(bits):
    L = emu_lib.lib()
    maxlen = 15 if bits == 4 else 7
    rng = random.Random(bits)
    alpha = "ACGTN" if bits == 4 else "ACGTN-."
    for n in range(1, 24):
        base = "".join(rng.choice(alpha) for _ in range(n + 2))
        seqs = [base]
        for j in range(n):                                     # the same allele (at offset 1) with symbol j changed
            t = list(base)
            t[1 + j] = alpha[(alpha.index(t[1 + j]) + 1) % len(alpha)]
            seqs.append("".join(t))
        if n >= 2:
            seqs.append(base[:-1])                             # the allele without its last symbol
        pool, offs = pool_bytes(seqs, bits)
        buf = C.create_string_buffer(pool, len(pool))
        sig0 = L.emu_make_sig(bits, buf, offs[0], len(seqs[0]), 0, 1, n)
        exact = L.emu_sig_exact(bits, sig0)
        assert bool(exact) == (n <= maxlen), n               # whole string in the signature up to maxlen symbols, a hash beyond
        for i, s in enumerate(seqs):
            ln = n if len(s) == n + 2 else n - 1
            same = s[1:1 + ln] == base[1:1 + n]
            sig = L.emu_make_sig(bits, buf, offs[i], len(s), 0, 1, ln)
            if exact or same:
                assert (sig == sig0) == same, (n, i)
            # allele_equal decides by the bases: equal iff the strings are
            assert bool(L.emu_allele_equal(bits, buf, offs[0], len(seqs[0]), 0, 1, n, offs[i], len(s), 0, 1, ln)) == same, (n, i)
            # on a reverse-strand record the allele is read through the complement: the same record on both sides is equal to itself
            assert L.emu_allele_equal(bits, buf, offs[i], len(s), 1, 1, ln, offs[i], len(s), 1, 1, ln) == 1
