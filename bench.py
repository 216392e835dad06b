#!/usr/bin/env python
"""bench.py — headline benchmark: assembly Mbp polished / second (BASELINE.json).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR]

One step = one pass of the polish hot path (classify -> CIGAR walk + pileup -> vote + compaction) over one
synthetic workload (default: BASELINE configs[1], one 5 Mbp contig at 100x, multi-mapped 150 bp pairs).
  value      whole-job Mbp/s with the packed inputs already resident in HBM (pp_polish_resident), device-timed
  e2e        the same metric through the reference-facing C-ABI call with HOST buffers (pp_polish): pinned-host
             H2D of the packed alignments and D2H of the polished bases inside the timed region
  roofline   the dominant kernel (k_tile: CIGAR walk + pileup + ordered depth + vote): algorithmic bytes / CUDA-event duration vs the measured HBM peak
  t3 / cli   the whole command from SAM text (pp_polish_files in a resident process / a fresh build/polypolish process)
  cpu_baseline  the CPU oracle (C++ restatement of the reference, 1 thread) on the same SAM text files (the whole
             workload when that is bounded - 5 Mbp x 100x: ~15 s - else a slice); `parity` compares its FASTA with the GPU's
With N > 1 (torchrun, one rank per GPU) the contigs of ONE config-5-shaped assembly (6.25 N contigs of 5 Mbp, repeat
families that cross contigs) shard across the ranks with no collective on the data path: every rank polishes its
shard, ghost records included (weak scaling); time = max over ranks.
--impl reference times the reference's CPU path (the oracle; the Rust reference cannot be built here) on rank 0.
K steps are timed on the kernel path and K on the e2e path.  The inputs are generated from fixed seeds, so they are the
same from run to run.
--dump-outputs DIR writes what the last timed step returned (rank 0's shard when N > 1) as DIR/<name>.npy, so that two
builds can be compared output for output; that step also copies its result to the host, outside the device-timed stages.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n_contigs per GPU, contig_len, depth)
    "5Mbp_x100": (1, 5_000_000, 100.0),      # BASELINE configs[1]
    "50kbp_x100": (1, 50_000, 100.0),        # configs[0]
    "5Mbp_x1000": (1, 5_000_000, 1000.0),    # configs[3]
    "500kbp_x100": (1, 500_000, 100.0),
    "6x5Mbp_x100": (6, 5_000_000, 100.0),    # one GPU's share of configs[4] (50 x 5 Mbp over 8 GPUs)
}
METRIC = "assembly Mbp polished/sec"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, device):
        self.device = device
        self.samples = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        sm, mx, reasons = [], None, set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes(arrs, G, out_len):
    """SURVEY.md §8(d): compulsory traffic of the canonical packed layout, each array counted once."""
    import numpy as np
    n = len(arrs["contig"])
    own = (arrs["flags"] & 4) == 0                       # records that carry their own SEQ
    seq_bytes = int(((arrs["seq_len"][own].astype(np.int64) + 1) // 2).sum())
    aln = 25 * n + 4 * len(arrs["cigar_ops"]) + seq_bytes
    return {"alignment_side": aln, "position_side": int(G + out_len), "total": int(aln + G + out_len)}


def _shm_dir(prefix, need_gb):
    import shutil
    shm = "/dev/shm"
    base = shm if os.path.isdir(shm) and shutil.disk_usage(shm).free > need_gb * (1 << 30) else None
    return tempfile.mkdtemp(prefix=prefix, dir=base)


def oracle_polish(fa, sams):
    """One run of the CPU oracle's whole `polish` command (C++ restatement of the reference, single thread like the
    reference) on SAM text that is already on disk / in the page cache.  Returns (seconds, result dict)."""
    from tests import oracle_lib
    o = oracle_lib.load()
    t0 = time.perf_counter()
    r = o.polish(fa, sams)
    return time.perf_counter() - t0, r


def reference_sample(workload):
    """What the CPU arm runs: the workload itself when one run of it is bounded (5 Mbp x 100x: ~15 s), else a slice."""
    n_c, clen, depth = WORKLOADS[workload]
    if n_c * clen * depth <= 6e8:
        return n_c, clen, depth, True
    clen = min(clen, 1_000_000)
    return 1, clen, (depth if clen * depth <= 6e8 else 100.0), False


DUMP_MAX_BYTES = 64_000_000
DUMP_FULL_BASES = 12_000_000        # up to this many polished bases are written whole (48 MB as float32)
DUMP_SAMPLE_BASES = 4_000_000       # above it, this many positions drawn with seed 0, and the positions (16 + 32 MB)


def dump_outputs(out_dir, sequences, changed, zero_depth, total_depth, n_aln_used):
    """Writes one polish result, as a caller of the polish call receives it, as float .npy files under out_dir:
    polished_bases (the ASCII codes of the polished contigs, concatenated), contig_offsets (where each contig starts in
    them, plus the total), changed, zero_depth and total_depth (per contig) and n_aln_used.  A result of more than
    DUMP_FULL_BASES bases is sampled at DUMP_SAMPLE_BASES fixed positions, written as polished_bases_index.
    All but total_depth are exact; the device sums total_depth in parallel, so it can differ in the last bits from run to
    run (include/pp_abi.h).  Returns the names written."""
    import numpy as np
    bases = np.frombuffer(b"".join(sequences), dtype=np.uint8)
    out = {"contig_offsets": np.cumsum([0] + [len(s) for s in sequences], dtype=np.int64).astype(np.float64),
           "changed": np.asarray(changed, dtype=np.float64), "zero_depth": np.asarray(zero_depth, dtype=np.float64),
           "total_depth": np.asarray(total_depth, dtype=np.float64), "n_aln_used": np.array([n_aln_used], dtype=np.float64)}
    if bases.size <= DUMP_FULL_BASES:
        out["polished_bases"] = bases.astype(np.float32)
    else:
        idx = np.sort(np.random.default_rng(0).choice(bases.size, DUMP_SAMPLE_BASES, replace=False))
        out["polished_bases"] = bases[idx].astype(np.float32)
        out["polished_bases_index"] = idx.astype(np.float64)
    if sum(a.nbytes for a in out.values()) > DUMP_MAX_BYTES:
        raise RuntimeError("bench: --dump-outputs would write more than %d bytes" % DUMP_MAX_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sorted(out)


def fasta_sequences(fasta):
    """The sequence lines of a polished FASTA (one header line and one sequence line per contig)."""
    return fasta.split(b"\n")[1::2]


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the host cores.  The Rust crate
    cannot be built in this image (no cargo/rustc; 78 un-vendored crates), so this is the oracle port, one thread (the
    reference has no threads).  Same config as the b200 arm's N=1 workload; the input files are generated once, outside
    the timed steps; one step = the whole `polish` command on them (page cache warm)."""
    if rank != 0:
        return
    import hashlib
    import shutil
    from polypolish_b200 import api
    n_c, clen, depth, same = reference_sample(args.workload)
    if world > 1:
        same = False         # the b200 arm's N > 1 workload is 6.25 N such contigs (config 5): one of them is the bounded CPU sample
    d = _shm_dir("pp_ref_", 6)
    try:
        syn = api.Synth(seed=2, n_contigs=n_c, contig_len=clen, depth=depth)
        fa, sams = syn.write(d)
        bp = syn.total_bp
        vals, sha = [], None
        for i in range(args.warmup + args.steps):
            dt, r = oracle_polish(fa, sams)
            sha = hashlib.sha256(r["fasta"]).hexdigest()
            if i >= args.warmup:
                vals.append((bp / 1e6 / dt, dt, r["secs"]))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, fasta_sequences(r["fasta"]), r["changed"], r["zero_depth"], r["total_depth"], r["used_total"])
    finally:
        shutil.rmtree(d, ignore_errors=True)
    v = sum(x[0] for x in vals) / len(vals)
    ms = 1e3 * sum(x[1] for x in vals) / len(vals)
    what = "the whole workload" if same else ("one contig of the %d-GPU workload's %d" % (world, (25 * world) // 4) if world > 1 else "a slice of the workload")
    sample = f"{bp} bp x {depth:g}x ({what}), whole `polish` command on page-cache-warm SAM text"
    line = {"metric": METRIC, "value": v, "unit": "Mbp/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u32 counters, f64 depth",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": args.workload, "same_config": same, "sample": sample, "fasta_sha256": sha},
            "cpu_baseline": {"value": v, "unit": "Mbp/s", "cores": 1, "kind": "port", "sample": sample, "phases_s": vals[-1][2]},
            "e2e": {"value": v, "unit": "Mbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="5Mbp_x100", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--wire4", action="store_true", help="e2e with the 4-bit arrays on the wire instead of the 2-bit format")
    ap.add_argument("--no-t3", action="store_true", help="skip the SAM-text-on-disk -> FASTA measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))

    import __graft_entry__ as g
    if rank == 0 or not os.path.exists(os.path.join(ROOT, "build", "libpolypolish_b200.so")):
        g.build()

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
    import polypolish_b200 as pp
    from polypolish_b200 import api

    n_c, clen, depth = WORKLOADS[args.workload]
    t0 = time.perf_counter()
    shard_info = None
    if world == 1:
        syn = api.Synth(seed=2, n_contigs=n_c, contig_len=clen, depth=depth)
        fasta = syn.fasta()
        packed = syn.pack(fasta)
        cview, aview = fasta.view, packed.view
        arrs = packed.arrays()
        G = int(fasta.off[-1])
        workload_name = args.workload
    else:
        # N > 1: BASELINE configs[4] - ONE assembly of 6.25 x N contigs of 5 Mbp (N = 8: the 50 contigs of config 5) at 100x with
        # repeat families that cross contigs, contig-sharded over the ranks (contig c -> rank c mod N).  Every rank generates the
        # reads of that one data set that have a record on its contigs (the generator's per-pair random streams make the subset
        # reproducible without the rest), runs the contig sharder on them (ghost records keep k across shards) and polishes
        # its shard.  No collective on the data path.
        n_total = (25 * world) // 4
        assign = [c % world for c in range(n_total)]
        syn = api.Synth(seed=5, n_contigs=n_total, contig_len=clen, depth=depth, cross_contig=0.01)
        syn.set_shard_filter(world, rank, assign)
        syn.set_threads(max(1, min(16, (os.cpu_count() or 8) // world)))     # (setup only: the same bytes whatever the count)
        fasta = syn.fasta()
        packed = syn.pack(fasta)
        shards = api.Shards(fasta.view, packed.view, world, shard_of_contig=assign, only_shard=rank)
        cview, aview, cmap, n_home = shards.get(rank)
        arrs = api.view_arrays(aview)
        n_c = cview.n_contigs
        G = int(np.ctypeslib.as_array(C.cast(cview.off, C.POINTER(C.c_uint64)), shape=(n_c + 1,))[-1])
        shard_info = {"contigs_total": n_total, "contigs_this_rank": n_c, "ghost_records_rank0": int(aview.n_aln - n_home)}
        workload_name = "config5_share_%dx5Mbp_x100_of_%d" % (n_c, n_total)
    t_gen = time.perf_counter() - t0

    ctx = pp.Context(local)
    # pinned copies of the packed arrays for the host-buffer (e2e) path
    L = pp.lib()
    pinned = []

    def pin(a):
        nbytes = max(1, a.nbytes)
        p = L.pp_host_alloc(nbytes)
        if not p:
            raise RuntimeError("pp_host_alloc failed")
        C.memmove(p, a.ctypes.data, a.nbytes)
        pinned.append(p)
        return p
    # The batch as it crosses PCIe: the 2-bit wire format of the packed arrays (pp_alignments_to_2bit - made once per batch on the host,
    # like the packing itself, outside the timed region; expanded to the kernels' 4-bit codes on the device inside it).
    wire_names = ["contig", "ref_start", "read_id", "seq_off", "seq_len", "cigar_off", "n_cigar", "nm", "flags", "cigar_ops", "seq_pool", "esc_pool"]
    t0 = time.perf_counter()
    two_bit = api.TwoBit(aview) if aview.seq_bits == 4 and not args.wire4 else None
    wire_prep_ms = (time.perf_counter() - t0) * 1e3 if two_bit else 0.0      # host pass, once per batch (word-parallel, up to 16 threads)
    wire_view = two_bit.view if two_bit else aview
    wire = api.view_arrays(wire_view)
    hv = api.Alignments()
    C.memmove(C.byref(hv), C.byref(wire_view), C.sizeof(api.Alignments))
    for name in wire_names:
        if getattr(wire_view, name) or name == "esc_pool":      # (cigar_off / read_id stay null in the 2-bit format: the device rebuilds them)
            setattr(hv, name, pin(wire[name]))
    h2d_bytes = sum(wire[n].nbytes for n in wire_names) + G + 8 * (n_c + 1)
    h2d_bytes_4bit = sum(arrs[n].nbytes for n in wire_names if n in arrs) + G + 8 * (n_c + 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- kernel path: inputs resident in HBM ----------------
    t0 = time.perf_counter()
    ctx.upload(cview, aview)                     # H2D of the packed arrays + the once-per-dataset position binning (k_bin, sort, k_permute*)
    upload_ms = (time.perf_counter() - t0) * 1e3
    for _ in range(args.warmup):
        r = ctx.polish_resident(fetch=False)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    t0 = time.perf_counter()
    stage = {}
    dev_ms = 0.0
    launches = 0
    dump = bool(args.dump_outputs) and rank == 0
    for i in range(args.steps):
        r = ctx.polish_resident(fetch=dump and i == args.steps - 1)
        dev_ms += r["timing"]["total_ms"]
        launches += r["timing"]["launches"]
        for k, v in r["timing"].items():
            if k.endswith("_ms"):
                stage[k] = stage.get(k, 0.0) + v
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    out_len = r["out_len"]
    ms_step = dev_ms / args.steps
    if dump:
        dump_outputs(args.dump_outputs, r["sequences"], r["changed"], r["zero_depth"], r["total_depth"], r["n_aln_used"])

    # ---------------- e2e: host buffers through pp_polish ----------------
    # (inputs in pinned host arrays, the result into caller-owned pinned buffers; the last result is checked against the
    #  kernel-path run above through its length and the library's own counters)
    out_res = ctx.pinned_result(n_c, G + G // 16 + (1 << 20))
    for _ in range(2):
        e = ctx.polish_packed(cview, hv, into=out_res)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    e2e_each = []
    for _ in range(e2e_steps):
        t1 = time.perf_counter()
        e = ctx.polish_packed(cview, hv, into=out_res)
        e2e_each.append((time.perf_counter() - t1) * 1e3)
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps
    e2e_median = sorted(e2e_each)[len(e2e_each) // 2]
    if int(e["out_len"]) != int(out_len):
        raise RuntimeError("e2e result length differs from the kernel-path result")
    d2h_bytes = int(e["out_len"]) + 8 * (3 * n_c + 1)
    ctx.free_pinned_result(out_res[1])
    clocks = sampler.stop() if rank == 0 else None      # sampled over both timed regions (kernel path + e2e)
    d2h_bytes = int(e["out_len"]) + 8 * (3 * n_c + 1)

    # ---------------- T3: the whole command, SAM/FASTA text on disk (page cache warm) -> polished FASTA bytes ----------------
    # ... and on the same files: the one-shot CLI process, the CPU oracle (cpu_baseline) and the parity check GPU == oracle.
    t3 = cli = cpu = parity = None
    if rank == 0 and world == 1:
        import hashlib
        import shutil
        full = G * depth <= 6e8                              # the whole workload as text is bounded (<= ~1.3 GB, oracle ~15 s)
        if full:
            tsyn, tdesc = syn, "the whole workload"
        else:
            tsyn = api.Synth(seed=2, contig_len=min(clen, 1_000_000), depth=min(depth, 100.0))
            tdesc = "a slice of the same generator"
        d = _shm_dir("pp_t3_", 6)
        try:
            fa_path, sam_paths = tsyn.write(d)
            tbp = int(tsyn.total_bp)
            sam_bytes = sum(os.path.getsize(x) for x in sam_paths)
            gpu_fasta = None
            if not args.no_t3:
                outs, best = {}, {}
                for mode, name, reps in ((0, "device_tokeniser", 4), (1, "host_packer", 2)):
                    ctx.set_parser(mode)
                    ts = []
                    for _ in range(reps):
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                        outs[name] = ctx.polish_files(fa_path, sam_paths)
                        ts.append((time.perf_counter() - t0) * 1e3)
                    best[name] = min(ts)
                ctx.set_parser(0)
                gpu_fasta = outs["device_tokeniser"]
                # the opt-in QUAL-stripping upload (pp_tok_set_strip_qual: 45 % fewer bytes over PCIe, paid for with a host pass over the text)
                ctx.set_strip_qual(1)
                ts = []
                for _ in range(3):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    outs["strip_qual"] = ctx.polish_files(fa_path, sam_paths)
                    ts.append((time.perf_counter() - t0) * 1e3)
                ctx.set_strip_qual(0)
                best["strip_qual"] = min(ts)
                rc_tok, tok_stats = ctx.tokenise(tsyn.fasta(), sam_paths)
                t3 = {"value": tbp / 1e6 / (best["device_tokeniser"] / 1e3), "unit": "Mbp/s", "ms": best["device_tokeniser"],
                      "host_packer_ms": best["host_packer"], "sam_text_bytes": int(sam_bytes), "files": len(sam_paths), "host_cores": os.cpu_count(),
                      "input": f"{tbp} bp x {depth:g}x ({tdesc})", "parsers_agree": outs["device_tokeniser"] == outs["host_packer"] == outs["strip_qual"],
                      "strip_qual_ms": best["strip_qual"],      # opt-in upload without the QUAL column: same bytes out; off by default unless this is the smaller number
                      "tokeniser": [{k: (round(v, 3) if isinstance(v, float) else v) for k, v in st.items()} for st in tok_stats],
                      "api": "pp_polish_files (FASTA + SAM paths in, FASTA bytes out), best of 4; host_packer = same call with pp_set_parser(1)"}
                # the drop-in command as a user runs it: a fresh process per call (CUDA start-up included)
                exe = os.path.join(ROOT, "build", "polypolish")
                if os.path.exists(exe):
                    ts, cli_out = [], None
                    for _ in range(3):
                        t0 = time.perf_counter()
                        pr = subprocess.run([exe, "polish", "--quiet", fa_path] + sam_paths, capture_output=True)
                        ts.append((time.perf_counter() - t0) * 1e3)
                        if pr.returncode != 0:
                            raise RuntimeError("build/polypolish polish failed: " + pr.stderr.decode()[-400:])
                        cli_out = pr.stdout
                    cli = {"value": tbp / 1e6 / (min(ts) / 1e3), "unit": "Mbp/s", "wall_ms": min(ts), "wall_ms_all": [round(x, 1) for x in ts],
                           "command": "build/polypolish polish --quiet draft.fasta reads_1.sam reads_2.sam > out.fasta (fresh process, page cache warm)",
                           "identical_to_library_call": cli_out == gpu_fasta}
            else:
                gpu_fasta = ctx.polish_files(fa_path, sam_paths)
            if not args.no_cpu_baseline:
                dt, orc = oracle_polish(fa_path, sam_paths)
                cpu = {"value": tbp / 1e6 / dt, "unit": "Mbp/s", "cores": 1, "kind": "port",
                       "sample": f"{tbp} bp x {depth:g}x ({tdesc}), whole `polish` command from the same SAM text files ({dt:.1f} s)",
                       "phases_s": orc["secs"]}
                parity = {"checked": True, "identical": orc["fasta"] == gpu_fasta, "sha256": hashlib.sha256(gpu_fasta).hexdigest(),
                          "oracle_sha256": hashlib.sha256(orc["fasta"]).hexdigest(), "bytes": len(gpu_fasta),
                          "what": f"polished FASTA of pp_polish_files vs the CPU oracle on the same files, {tbp} bp x {depth:g}x ({tdesc})"}
                if cli is not None:
                    parity["cli_identical"] = cli_out == orc["fasta"]
            ctx.upload(cview, aview)
        finally:
            shutil.rmtree(d, ignore_errors=True)

    # ---------------- max over ranks ----------------
    t = torch.tensor([ms_step, wall_ms / args.steps, e2e_ms], dtype=torch.float64, device=f"cuda:{local}")
    tot = torch.tensor([float(G), float(h2d_bytes), float(d2h_bytes), float(aview.n_aln)], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms_step_max, wall_step_max, e2e_ms_max = t.tolist()
    total_bp, h2d_total, d2h_total, aln_total = tot.tolist()   # the whole job: every rank's contigs

    if rank == 0:
        hbm, how = peaks()
        ab = algorithmic_bytes(arrs, G, out_len)
        sc_ms = stage["tile_ms"] / args.steps
        k_bytes = ab["alignment_side"] + G                 # what one k_tile launch must move: every alignment record, CIGAR op and read base, and the draft
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic = tj.get(args.workload) if world == 1 else None
            traffic_src = "static, from profiles/traffic.json (%s); not measured in this run" % tj.get("source", "ncu --set full capture")
        line = {
            "metric": METRIC, "value": total_bp / 1e6 / (ms_step_max / 1e3), "unit": "Mbp/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step_max, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8 bases / u32 counters / f64 depth", "data": "synthetic",
            "config": {"workload": workload_name, "contigs_rank0": n_c, "contig_bp": clen, "depth": depth, "assembly_bp": int(total_bp),
                       "reads": "150 bp paired, multi-mapped (repeat families x7,x5,x3,x2,x4" + (", plus families that cross contigs)" if world > 1 else ")"),
                       "alignments_rank0": int(aview.n_aln), "alignments_total": int(aln_total), "sharding": shard_info,
                       "parallelism": (f"one assembly, contigs sharded over {world} ranks by pp_shards_build_assigned (ghost records), no collective on the data path"
                                       if world > 1 else "1 GPU"),
                       "timing": "CUDA events on the library stream, max over ranks",
                       "cache": "inputs (%.0f MB packed) larger than the 126 MB L2" % (h2d_bytes / 1e6)},
            "e2e": {"value": total_bp / 1e6 / (e2e_ms_max / 1e3), "unit": "Mbp/s", "ms_per_step": e2e_ms_max,
                    "h2d_bytes_per_step": int(h2d_total), "d2h_bytes_per_step": int(d2h_total), "api": "pp_polish (host SoA in, host bases out)",
                    "wire": ("2-bit read bases, cigar_off and read_id rebuilt on the device (pp_alignments_to_2bit once per batch, outside the timed region like the packing; %d B/step as 4-bit)" % h2d_bytes_4bit
                             if two_bit else "%d-bit read bases" % aview.seq_bits),
                    "wire_prep_ms_rank0": round(wire_prep_ms, 1),     # pp_alignments_to_2bit on the host, once per batch, NOT inside ms_per_step (like the packing that makes the arrays)
                    "ms_per_step_median_rank0": round(e2e_median, 3),     # (a shared box can stall single H2D copies; the value above is the mean)
                    "last_step_ms": {k: round(v, 3) for k, v in e["timing"].items() if k.endswith("_ms") and v}},   # h2d = upload + position binning
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "k_tile<4>", "achieved": k_bytes / 1e9 / (sc_ms / 1e3), "peak": hbm,
                         "unit": "GB/s", "frac": k_bytes / 1e9 / (sc_ms / 1e3) / hbm, "traffic": traffic, "traffic_source": traffic_src, "peak_source": how,
                         "algorithmic_bytes_per_launch": k_bytes, "kernel_ms": sc_ms,
                         "whole_path": {"algorithmic_bytes": ab["total"], "ms": ms_step, "achieved": ab["total"] / 1e9 / (ms_step / 1e3),
                                        "frac": ab["total"] / 1e9 / (ms_step / 1e3) / hbm}},
            "stages_ms": {k: v / args.steps for k, v in sorted(stage.items())},
            "wall_ms_per_step": wall_step_max, "clocks": clocks, "setup_s": t_gen,
            "dataset_upload_ms": upload_ms,     # pageable H2D + binning, once per dataset; `value` times pp_polish_resident on the binned dataset, `e2e` (pp_polish) pays for both every step
        }
        if t3 is not None:
            line["t3"] = t3
        if cli is not None:
            line["cli"] = cli
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if parity is not None:
            line["parity"] = parity
        print(json.dumps(line), flush=True)
        if parity is not None and not (parity["identical"] and parity.get("cli_identical", True)):
            raise SystemExit("bench: the GPU FASTA differs from the CPU oracle's on the same input (parity broken)")
    for p in pinned:
        L.pp_host_free(p)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)
    main()
