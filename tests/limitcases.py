"""Deterministic edge-case builders for the polish kernels' fallback and boundary paths (polypolish_b200/csrc/polish_dev.cuh,
polish_kernels.cu).  Every builder returns (fuzzgen.Case, info): FASTA and SAM texts, the options to polish with, and the quantities
that show which size threshold the case crosses, so a test can assert the path it is meant to reach was reached.

`scale` is "emu" (small enough for the CPU emulator of the kernels) or "gpu" (the size that crosses the device threshold; a few
thresholds are the same at both scales because the emulator runs the same device code with the same constants).  Reads are built
by walking the draft, as fuzzgen does, so every CIGAR consumes exactly its SEQ.
"""
import os
import random
import re

from tests import fuzzgen

# The constants of polish_dev.cuh / polish_kernels.cu the cases are sized against, read from the sources: when one changes, the
# "path ran" assertions of the tests follow it (and fail if a case no longer crosses its threshold) instead of going stale.
_CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "polypolish_b200", "csrc")


def _defines(*files):
    out = {}
    for f in files:
        for m in re.finditer(r"^#define\s+(\w+)\s+([^/\n]+)", open(os.path.join(_CSRC, f)).read(), re.M):
            expr = re.sub(r"\b(\d+)u\b", r"\1", m.group(2).strip())
            try:
                out[m.group(1)] = int(eval(expr, {}, dict(out)))
            except Exception:
                pass
    return out


_D = _defines("polish_dev.cuh", "polish_kernels.cu")
TL_T = _D["TL_T"]                            # positions per tile / compaction chunk
PP_BIN = _D["PP_BIN"]                        # binning granularity (a tile looks back ceil(max_ext / PP_BIN) bins)
TL_FAST_LEN = _D["TL_FAST_LEN"]              # longest read of the register fast path
TL_LONG_E = _D["TL_LONG_E"]                  # alignments with more entries go to the long list
TL_QCAP = _D["TL_QCAP"]                      # queued (deferred) reads per tile
SC_GROUP_SCAN_LIMIT = _D["SC_GROUP_SCAN_LIMIT"]   # records of one read group k_goodk scans outside its block
PR_THREADS = _D["PR_THREADS"]                # k_goodk block
CP_STAGE = _D["CP_STAGE"]                    # output bytes k_compact stages in shared memory per chunk
PP_INIT_IMAGE = _D["PP_INIT_IMAGE"]          # per-call reset block that travels as one copy
MAX_U16 = 0xFFFF

IUPAC = "RYSWKMBVDHN"
DEFAULT_OPTS = dict(fraction_invalid=0.2, fraction_valid=0.5, max_errors=10, min_depth=5, careful=False)


def _r256(n):
    return (n + 255) & ~255


def reset_block_bytes(n_contigs, n_reads, global_k):
    """Size of the per-call reset block of run_polish (polish_kernels.cu:400-405): changed, zero_depth, total_depth per contig,
    DevStatus (48 B), the global-k counts, DevParams (32 B), each rounded to 256 B.  Above PP_INIT_IMAGE it is reset by memsets."""
    return 3 * _r256(8 * n_contigs) + _r256(48) + _r256((n_reads + 1) * 4 if global_k else 4) + _r256(32)


def first_node_cap(n_aln, G):
    """The node pool's first guess (polish_kernels.cu:280)."""
    return min(0x7FFFFFFF, max(1 << 16, n_aln // 8 + G // 64))


def first_out_cap(G):
    """The output buffer's first guess on the device (polish_kernels.cu:281)."""
    return G + G // 16 + (1 << 20)


def rand_seq(rng, n, alphabet="ACGT"):
    return "".join(rng.choice(alphabet) for _ in range(n))


def cigar_of(ops):
    return "".join(f"{n}{op}" for op, n in ops)


def spec_read(draft, start, spec):
    """A read from an explicit walk of the draft: spec items ("M", n), ("M", n, {offset: base}), ("D", n), ("I", bases).
    Returns (cigar, seq, nm, ref_span)."""
    ops, seq, nm, p = [], [], 0, start
    for item in spec:
        op = item[0]
        if op == "M":
            n, subs = item[1], (item[2] if len(item) > 2 else {})
            for t in range(n):
                b = subs.get(t, draft[p + t])
                nm += b != draft[p + t]
                seq.append(b)
            ops.append(("M", n)); p += n
        elif op == "D":
            ops.append(("D", item[1])); nm += item[1]; p += item[1]
        else:
            ops.append(("I", len(item[1]))); seq.extend(item[1]); nm += len(item[1])
    ops = fuzzgen.merge_ops(ops)
    assert p <= len(draft), (start, spec)
    return cigar_of(ops), "".join(seq), nm, p - start


def walk_read(rng, draft, edits, start, want_len, apply=0.9):
    """fuzzgen.build_read: walk the draft from `start`, applying the per-position truth edits (sub / del / ins) with probability
    `apply`, until the read has `want_len` bases.  Returns (cigar, seq, nm, ref_span)."""
    ops, read, nm, p = [], [], 0, start
    while len(read) < want_len and p < len(draft):
        e = edits.get(p) if rng.random() < apply else None
        base = draft[p]
        if e is None or (e[0] == "del" and not ops):
            ops.append(("M", 1)); read.append(base)
        elif e[0] == "sub":
            ops.append(("M", 1)); read.append(e[1]); nm += e[1] != base
        elif e[0] == "del":
            ops.append(("D", 1)); nm += 1
        else:
            ops.append(("M", 1)); read.append(base)
            ops.append(("I", len(e[1]))); read.extend(e[1]); nm += len(e[1])
        p += 1
    ops = fuzzgen.merge_ops(ops)
    while ops and ops[-1][0] in "DI":                       # end on a match
        op, n = ops.pop()
        if op == "I":
            del read[-n:]
        else:
            p -= n
    return cigar_of(ops), "".join(read), nm, p - start


def truth_edits(rng, L, rate, lo=5, hi=None, ins_len=(1, 3)):
    hi = L - 5 if hi is None else hi
    edits = {}
    for i in range(lo, hi):
        r = rng.random()
        if r < rate * 0.5:
            edits[i] = ("sub", rng.choice("ACGT"))
        elif r < rate * 0.75:
            edits[i] = ("del",)
        elif r < rate:
            edits[i] = ("ins", rand_seq(rng, rng.randint(*ins_len)))
    return edits


def parse_cigar(cigar):
    ops, n = [], ""
    for ch in cigar:
        if ch.isdigit():
            n += ch
        else:
            ops.append((ch, int(n))); n = ""
    return ops


def entries_of(cigar, seq):
    """(reference offset, allele) of every entry the alignment adds after the right-end trim (alignment.rs:175-201, 364-378)."""
    rb, i = [], 0
    for op, n in parse_cigar(cigar):
        for _ in range(n):
            if op in "M=X":
                rb.append([i, i + 1]); i += 1
            elif op == "I":
                rb[-1][1] = i + 1; i += 1
            elif op == "D":
                rb.append([i, i])
    assert i == len(seq), (cigar, len(seq))
    last = seq[rb[-1][0]:rb[-1][1]]
    while rb and seq[rb[-1][0]:rb[-1][1]] == last:
        rb.pop()
    if rb:
        rb.pop()
    return [(t, "-" if a == b else seq[a:b]) for t, (a, b) in enumerate(rb)]


class Sam:
    """SAM text under construction; QNAMEs are consecutive records (one read group each)."""

    def __init__(self, contigs):
        self.lines = ["@HD\tVN:1.6\tSO:unsorted"] + [f"@SQ\tSN:{n}\tLN:{len(s)}" for n, s in contigs]
        self.n_records = 0
        self.groups = 0
        self._last_q = None

    def rec(self, qname, flag, rname, pos0, cigar, seq, nm, tags=()):
        if qname != self._last_q:
            self.groups += 1
            self._last_q = qname
        self.lines.append("\t".join([qname, str(flag), rname, str(pos0 + 1), "60", cigar, "*", "0", "0", seq, "*", f"NM:i:{nm}"] + list(tags)))
        self.n_records += 1

    def text(self):
        return "\n".join(self.lines) + "\n"


def fasta_text(contigs, width=80):
    out = []
    for n, s in contigs:
        out.append(">" + n)
        out.extend(s[i:i + width] for i in range(0, len(s), width))
    return "\n".join(out) + "\n"


def make_case(contigs, sams, **opts):
    o = dict(DEFAULT_OPTS)
    o.update(opts)
    return fuzzgen.Case(fasta_text(contigs), [s.text() for s in sams], o)


# ---------------------------------------------------------------------------------------------------------------------------------
def long_reads(scale="emu", seed=1):
    """Reads longer than the fast path: exactly 192/193/256/257/512/513 reference entries (M only, with a deletion, with an
    insertion), 2-5 kbp (emu) or 2-20 kbp (gpu) reads with indels, one read of exactly 65,535 bases, both strands, starts and ends on
    tile (2048) and bin (256) borders, and multi-mapped reads (k = 3 with SEQ=* secondaries) over them, so that the ordered depth walk
    merges three bins and the long list (depth_walk_steps)."""
    rng = random.Random(seed)
    L1, L2 = (66_000, 9_000) if scale == "emu" else (72_000, 30_000)
    c1, c2 = rand_seq(rng, L1), rand_seq(rng, L2)
    contigs = [("big", c1), ("side", c2)]
    ed1, ed2 = truth_edits(rng, L1, 0.01), truth_edits(rng, L2, 0.01)
    sam = Sam(contigs)
    info = dict(E=[], k=set(), max_len=0)
    n = [0]

    def add(rname, draft, start, spec, strand, secondaries=0):
        cigar, seq, nm, span = spec_read(draft, start, spec)
        q = f"r{n[0]}"
        n[0] += 1
        sam.rec(q, 16 if strand else 0, rname, start, cigar, seq, min(nm, 10))
        info["E"].append(span)
        info["max_len"] = max(info["max_len"], len(seq))
        for j in range(secondaries):                         # SEQ=* secondaries with the same CIGAR elsewhere on `side`
            st = rng.randint(0, L2 - span - 1)
            sam.rec(q, 256 | (16 if (strand ^ (j & 1)) else 0), "side", st, cigar, "*", rng.randint(0, 6))
        if secondaries:
            info["k"].add(1 + secondaries)

    for E in (192, 193, 256, 257, 512, 513):
        for start in (2 * TL_T, 3 * TL_T - E, 5 * PP_BIN, 9 * PP_BIN - E, 7 * PP_BIN + 3):
            for dup in range(6):
                strand = dup & 1
                sec = 2 if dup % 3 == 0 else 0               # k = 3: 1/3 is not dyadic
                add("big", c1, start, [("M", E, {E // 2: "ACGT"[(dup + E) % 4]} if dup < 4 else {})], strand, sec)
                d = 1 + dup                                  # same number of entries with a deletion / an insertion inside
                add("big", c1, start, [("M", E // 3), ("D", d), ("M", E - E // 3 - d)], strand, sec)
                add("big", c1, start, [("M", E // 3), ("I", rand_seq(rng, 2)), ("M", E - E // 3)], strand, 0)
    lens = (2000, 3000, 5000) if scale == "emu" else (2000, 5000, 11_000, 20_000)
    for length in lens:
        for dup in range(7):
            start = rng.choice([0, TL_T, 4 * TL_T, rng.randint(0, L1 - length - 100)])
            cigar, seq, nm, span = walk_read(rng, c1, ed1, start, length)
            q = f"r{n[0]}"
            n[0] += 1
            sam.rec(q, 16 if dup & 1 else 0, "big", start, cigar, seq, min(nm, 10))
            info["E"].append(span)
            info["max_len"] = max(info["max_len"], len(seq))
            if dup % 2 == 0:
                for j in range(2):
                    st = rng.randint(0, L1 - span - 1)
                    sam.rec(q, 256 | (16 if j else 0), "big", st, cigar, "*", rng.randint(0, 6))
                info["k"].add(3)
    # the longest read the packed layout holds (u16 seq_len): 65,535 bases from position 0, plus short reads on the side contig
    cigar, seq, nm, span = spec_read(c1, 100, [("M", 30_000), ("D", 3), ("M", 20_000), ("I", "ACG"), ("M", MAX_U16 - 50_003)])
    sam.rec("huge", 0, "big", 100, cigar, seq, nm)
    info["E"].append(span)
    info["max_len"] = max(info["max_len"], len(seq))
    for _ in range(L2 * 8 // 150):
        start = rng.randint(0, L2 - 160)
        cigar, seq, nm, span = walk_read(rng, c2, ed2, start, 150)
        sam.rec(f"s{n[0]}", rng.choice([0, 16]), "side", start, cigar, seq, min(nm, 10))
        n[0] += 1
    info["max_binned_E"] = max(e for e in info["E"] if e <= TL_LONG_E)
    info["n_long"] = sum(1 for e in info["E"] if e > TL_LONG_E)
    info["k"] = sorted(info["k"])
    return make_case(contigs, [sam]), info


def one_indel_bounds(scale="emu", seed=2):
    """aM bI|bD cM reads at the edges of the two-segment fast walk (TR_FAST1, polish_dev.cuh:335-341): a in {255, 256},
    b in {1, 4095, 4096}, c in {8, 9} (all longer than the fast path, so general walks), and the edges that do decide TR_FAST1:
    read length 192 / 193, entries 512 / 513, last run 8 / 9, a of 1, homopolymer tails of 7 / 8 bases in the last run."""
    rng = random.Random(seed)
    L = 6_000
    draft = list(rand_seq(rng, L))
    tails = {}
    for i, t in enumerate((7, 8, 7, 8)):                     # homopolymer runs the reads can end on
        p = 5200 + 150 * i
        draft[p:p + t] = "ACGT"[i] * t
        draft[p - 1] = "C" if i != 1 else "A"
        draft[p + t] = "G" if i != 2 else "T"
        tails[p + t] = t
    draft = "".join(draft)
    sam = Sam([("ctg", draft)])
    info = dict(n_fast1=0, n_one_indel=0)
    n = [0]

    def add(start, spec, reps=6):
        for r in range(reps):
            subs = {} if r < 4 else {1: "ACGT"[r % 4]}
            sp = [(spec[0][0], spec[0][1], subs)] + list(spec[1:])
            cigar, seq, nm, span = spec_read(draft, start, sp)
            sam.rec(f"q{n[0]}", 16 if r & 1 else 0, "ctg", start, cigar, seq, min(nm, 10))
            n[0] += 1
            a, mid, c = spec[0][1], spec[1], spec[2][1]
            b = mid[1] if mid[0] == "D" else len(mid[1])
            E = a + c + (b if mid[0] == "D" else 0)
            fast1 = len(seq) <= TL_FAST_LEN and E <= TL_LONG_E and 1 <= a <= 255 and 1 <= b <= 4095 and c >= 9
            info["n_one_indel"] += 1
            info["n_fast1"] += fast1

    st = 0
    for a in (255, 256):
        for b in (1, 4095, 4096):
            for c in (8, 9):
                add(st, [("M", a), ("D", b), ("M", c)])
                add(st + 7, [("M", a), ("I", rand_seq(rng, b)), ("M", c)], reps=6 if b < 4095 else 3)
                st += 60
    # the edges that decide TR_FAST1 (len <= 192, E <= 512, a >= 1, c >= 9)
    for (a, c) in ((100, 92), (100, 93), (1, 191), (183, 9), (184, 8)):
        add(st, [("M", a), ("D", TL_LONG_E - a - c), ("M", c)])          # E = 512
        add(st + 20, [("M", a), ("D", TL_LONG_E + 1 - a - c), ("M", c)])  # E = 513
        add(st + 40, [("M", a), ("I", rand_seq(rng, 2)), ("M", c - 2)])   # length a + c
        st += 60
    st = 3_000
    for a in (40, 120):
        for b in (1, 3):
            for c in (8, 9, 30):
                add(st, [("M", a), ("I", rand_seq(rng, b)), ("M", c)])
                add(st + 30, [("M", a), ("D", b), ("M", c)])
                st += 60
    for end, t in tails.items():                             # last run ends on a homopolymer of 7 / 8 bases
        for c in (9, 12):
            add(end - c - 1 - 60, [("M", 60), ("D", 1), ("M", c)])
            add(end - c - 60, [("M", 60), ("I", "T"), ("M", c)])
    return make_case([("ctg", draft)], [sam]), info


def queue_overflow(scale="emu", seed=3, seq_bits=4):
    """More than TL_QCAP reads that are not plain fast walks in one tile, all starting inside it: the queue overflows and the
    rest are walked in place inside the chunk loop.  seq_bits=4: reads with two or more indels; seq_bits=8: plain reads, plus one
    '.' in one read's SEQ, which puts the whole batch in the 8-bit pool, where no read takes the fast walk."""
    rng = random.Random(seed)
    L = 3_000
    draft = rand_seq(rng, L)
    edits = truth_edits(rng, L, 0.05 if seq_bits == 4 else 0.01, ins_len=(1, 2))
    if seq_bits == 8:
        edits = {p: e for p, e in edits.items() if e[0] == "sub"}
    sam = Sam([("ctg", draft)])
    n_reads = 1_150
    info = dict(deferred_in_tile0=0)
    while sam.n_records < n_reads:
        start = rng.randint(0, TL_T - 150)
        cigar, seq, nm, span = walk_read(rng, draft, edits, start, rng.randint(60, 140))
        ops = parse_cigar(cigar)
        if seq_bits == 4 and sum(1 for op, _ in ops if op in "ID") < 2:
            continue
        if nm > 10:
            continue
        q = f"q{sam.n_records}"
        sam.rec(q, rng.choice([0, 16]), "ctg", start, cigar, seq, nm)
        info["deferred_in_tile0"] += 1
        if rng.random() < 0.2:                               # a SEQ=* secondary in the same tile: k = 2, the ordered depth walk
            sam.rec(q, 256 | rng.choice([0, 16]), "ctg", rng.randint(0, TL_T - span - 1), cigar, "*", rng.randint(0, 5))
            info["deferred_in_tile0"] += 1
    if seq_bits == 8:                                        # one byte outside the 16 BAM letters
        i = next(j for j in range(len(sam.lines) - 500, 0, -1) if sam.lines[j].split("\t")[9] != "*")
        f = sam.lines[i].split("\t")
        f[9] = f[9][:20] + "." + f[9][21:]
        sam.lines[i] = "\t".join(f)
    for _ in range(200):                                     # ordinary coverage of the second tile
        start = rng.randint(TL_T, L - 150)
        cigar, seq, nm, span = walk_read(rng, draft, edits, start, 100)
        sam.rec(f"t{sam.n_records}", 0, "ctg", start, cigar, seq, min(nm, 10))
    return make_case([("ctg", draft)], [sam]), info


def big_group(scale="emu", seed=4, n_records=9_000, many_reads=False):
    """One QNAME with n_records records: one primary with the SEQ, the rest SEQ=* secondaries over a repeat family on both strands,
    good and bad ones mixed (soft clips, NM above max_errors, ZP:Z:fail), so that k depends on the options.  The group starts
    mid-block (not on a multiple of 256 records).  It is larger than the SC_GROUP_SCAN_LIMIT records k_goodk scans outside its block:
    FL_BIGGROUP, then k_classify_multi + k_goodk<true>.  many_reads: more than 16,200 other read groups, so that the global-k
    counts make the per-call reset block larger than PP_INIT_IMAGE (reset by memsets)."""
    rng = random.Random(seed)
    unit = rand_seq(rng, 300)
    copies = 30
    rep = "".join("".join(b if rng.random() > 0.02 else rng.choice("ACGT") for b in unit) for _ in range(copies))
    uniq = rand_seq(rng, 3_000)
    contigs = [("rep", rep), ("uniq", uniq)]
    ed = truth_edits(rng, len(uniq), 0.01)
    sam = Sam(contigs)
    n_bg = 17_000 if many_reads else 1_800
    bg_len = 50 if many_reads else 100
    pre = 300                                                # records before the group: it starts at 300 % 256 = 44 in its block

    def background(i):
        if rng.random() < 0.7:
            start = rng.randint(0, len(uniq) - bg_len - 10)
            cigar, seq, nm, span = walk_read(rng, uniq, ed, start, bg_len)
            sam.rec(f"b{i}", rng.choice([0, 16]), "uniq", start, cigar, seq, min(nm, 10))
        else:
            start = rng.randint(0, len(rep) - bg_len)
            sam.rec(f"b{i}", rng.choice([0, 16]), "rep", start, f"{bg_len}M", rep[start:start + bg_len], 0)

    for i in range(pre):
        background(i)
    rl = 100
    off = rng.randint(0, 300 - rl)
    p0 = 7 * 300 + off
    primary = rep[p0:p0 + rl]
    group_start = sam.n_records
    sam.rec("big", 0, "rep", p0, f"{rl}M", primary, 0)
    good = {"default": 1, "max_errors=2": 1}
    for j in range(n_records - 1):
        c = rng.randrange(copies)
        st = c * 300 + off + rng.randint(-3, 3) if c * 300 + off + 3 + rl <= len(rep) and c * 300 + off >= 3 else c * 300 + off
        rev = rng.random() < 0.03
        kind = rng.random()
        tags = []
        if kind < 0.08:
            cg, nm = f"5S{rl - 5}M", rng.randint(0, 4)       # soft clip: not good
        elif kind < 0.16:
            cg, nm = f"{rl}M", rng.randint(11, 40)           # NM above the default max_errors
        elif kind < 0.24:
            cg, nm, tags = f"{rl}M", rng.randint(0, 4), ["ZP:Z:fail"]
        else:
            cg, nm = f"{rl}M", rng.randint(0, 8)
        g = cg.endswith("M") and not cg.startswith("5S") and not tags
        good["default"] += g and nm <= 10
        good["max_errors=2"] += g and nm <= 2
        sam.rec("big", 256 | (16 if rev else 0), "rep", st, cg, "*", nm, tags)
    for i in range(pre, n_bg):
        background(i)
    info = dict(group_size=n_records, group_start=group_start, good=good, n_reads=sam.groups, n_contigs=2,
                reset_bytes=reset_block_bytes(2, sam.groups, True))
    return make_case(contigs, [sam]), info


def many_contigs(scale="emu", seed=5):
    """Thousands of short contigs (1, 2, 7, 8, 9, 31, 127, 128, 129, 300 bp): one warp's 128 positions and one k_compact thread's 8
    positions hold several contigs (per-contig statistics, out_off), and above ~2,700 contigs the per-call reset block no longer
    fits PP_INIT_IMAGE.  Reads inside the contigs, some from end to end, a few multi-mapped (k = 2); draft errors on every contig
    of 7 bp or more are corrected."""
    rng = random.Random(seed)
    n = 400 if scale == "emu" else 3_000
    sizes = (1, 2, 7, 8, 9, 31, 127, 128, 129, 300)
    contigs = []
    for i in range(n):
        L = sizes[i % len(sizes)] if i < 2 * len(sizes) else rng.choice(sizes)
        contigs.append((f"c{i}", rand_seq(rng, L)))
    sam = Sam(contigs)
    q = 0
    by_len = {}
    for name, s in contigs:
        by_len.setdefault(len(s), []).append(name)
    seqs = dict(contigs)
    for name, s in contigs:
        L = len(s)
        subs = {}
        if L >= 7:
            for p in sorted({L // 2, L // 3, rng.randrange(1, L - 3)}):
                subs[p] = rng.choice([b for b in "ACGT" if b != s[p]])
        truth = "".join(subs.get(i, b) for i, b in enumerate(s))
        for r in range(6):                                   # end to end
            sam.rec(f"f{q}", 16 if r & 1 else 0, name, 0, f"{L}M", truth, min(10, len(subs)))
            q += 1
        for r in range(3 if L >= 8 else 1):                  # inside
            a = rng.randrange(0, L)
            b = rng.randrange(a + 1, L + 1)
            sam.rec(f"p{q}", rng.choice([0, 16]), name, a, f"{b - a}M", truth[a:b], sum(1 for i in subs if a <= i < b))
            q += 1
        if L >= 8 and rng.random() < 0.3:                    # a second hit on another contig of the same length: k = 2
            other = rng.choice(by_len[L])
            sam.rec(f"m{q}", 0, name, 0, f"{L}M", truth, len(subs))
            sam.rec(f"m{q}", 256, other, 0, f"{L}M", "*", sum(1 for i, b in enumerate(truth) if b != seqs[other][i]))
            q += 1
    offs, G = [], 0
    for _, s in contigs:
        offs.append(G)
        G += len(s)
    groups8 = {}
    for o in offs:
        groups8[o // 8] = groups8.get(o // 8, 0) + 1
    info = dict(n_contigs=n, G=G, reset_bytes=reset_block_bytes(n, sam.groups, False),
                max_contigs_in_8=max(groups8.values()), n_short=sum(1 for _, s in contigs if len(s) < 128))
    return make_case(contigs, [sam]), info


def other_allele_flood(scale="emu", seed=6):
    """More distinct (position, allele) pairs than the node pool's first guess, max(65,536, n_aln/8 + G/64) (polish_kernels.cu:280):
    a ~20 kbp contig at ~30x, reads full of random IUPAC letters and short distinct insertions.  The device sets FL_NODE_OVF,
    grows the pool and repeats the call."""
    rng = random.Random(seed)
    L = 3_000 if scale == "emu" else 20_000
    draft = rand_seq(rng, L)
    sam = Sam([("ctg", draft)])
    distinct = set()
    n_reads = L * 30 // 150
    for i in range(n_reads):
        start = rng.randint(0, L - 170)
        spec, p = [], 0
        while p < 150:
            run = rng.randint(3, 12)
            subs = {t: rng.choice(IUPAC) for t in range(run) if rng.random() < 0.2}
            spec.append(("M", run, subs))
            p += run
            if rng.random() < 0.6 and p < 140:
                spec.append(("I", rand_seq(rng, rng.randint(1, 3), "ACGTN")))
        cigar, seq, nm, span = spec_read(draft, start, spec)
        sam.rec(f"q{i}", rng.choice([0, 16]), "ctg", start, cigar, seq, nm)
        for t, a in entries_of(cigar, seq):
            if a not in ("A", "C", "G", "T", "-"):
                distinct.add((start + t, a))
    info = dict(distinct_other=len(distinct), n_aln=n_reads, G=L, first_node_cap=first_node_cap(n_reads, L))
    return make_case([("ctg", draft)], [sam], max_errors=1_000), info


def long_insertions(scale="emu", seed=7, seq_bits=4):
    """Insertions around the exact-signature limit (4-bit pool: alleles of 15 / 16 symbols = insertions of 14-17 bases; 8-bit pool:
    alleles of 7 / 8 bytes = insertions of 6-9 bytes), alleles that agree in every symbol but the last, enough support for some
    to win; a chunk whose output exceeds k_compact's shared-memory stage (unstaged compaction); at gpu scale more voted-in
    inserted bases than the first output buffer, G + G/16 + 1 MiB (device repeat, then the caller's retry).  The 8-bit variant
    puts '-' bytes inside inserted alleles: they are dropped from the output (polish.rs:188)."""
    rng = random.Random(seed)
    n_big, big_len = (20, 300) if scale == "emu" else (400, 3_000)
    spacing = 10
    lens = (14, 15, 16, 17) if seq_bits == 4 else (6, 7, 8, 9)
    L = spacing * (TL_T // spacing + 4 + n_big) + 200
    draft = rand_seq(rng, L)
    sam = Sam([("ctg", draft)])
    info = dict(voted_in=0, chunk_bytes={})
    q = [0]
    alpha = "ACGT" if seq_bits == 4 else "ACGT-"

    def site(i, alleles):
        """Reads 5M <ins> 5M around site i (its M base at 10 i + 9); `alleles` = list of (insertion, number of reads)."""
        p = spacing * i + 9
        for ins, cnt in alleles:
            for r in range(cnt):
                cigar, seq, nm, span = spec_read(draft, p - 4, [("M", 5), ("I", ins), ("M", 5)])
                sam.rec(f"q{q[0]}", 16 if r & 1 else 0, "ctg", p - 4, cigar, seq, min(nm, 10))
                q[0] += 1
        return p

    def ins_of(n, alphabet=alpha):
        s = rand_seq(rng, n, alphabet)
        if seq_bits == 8 and "-" not in s[1:-1]:
            s = s[0] + "-" + s[2:]
        return s

    def won(p, ins):                                         # a site whose one allele wins: the draft base + the insertion
        kept = len(ins.replace("-", ""))
        info["voted_in"] += kept
        info["chunk_bytes"][p // TL_T] = info["chunk_bytes"].get(p // TL_T, 0) + 1 + kept

    i = 0
    for n in lens:
        a = ins_of(n)
        b = a[:-1] + ("A" if a[-1] != "A" else "C")          # differs only in the last symbol
        for alleles in ([(a, 6)], [(a, 6), (b, 3)], [(a, 3), (b, 3)], [(a, 5), (b, 1)], [(b, 6)]):
            p = site(i, alleles)
            i += 1
            if len(alleles) == 1:
                won(p, alleles[0][0])
    i = max(i, TL_T // spacing + 4)                          # the long ones after the first chunk: their chunk's output starts past 0
    for _ in range(n_big):
        ins = ins_of(big_len, "ACGT")                       # (8-bit: one '-' inside)
        won(site(i, [(ins, 6)]), ins)
        i += 1
    info["G"] = L
    info["max_chunk_bytes"] = max(info["chunk_bytes"].values())
    return make_case([("ctg", draft)], [sam]), info


BUILDERS = dict(long_reads=long_reads, one_indel_bounds=one_indel_bounds, queue_overflow=queue_overflow, big_group=big_group,
                many_contigs=many_contigs, other_allele_flood=other_allele_flood, long_insertions=long_insertions)
