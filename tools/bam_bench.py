#!/usr/bin/env python
"""BAM against SAM input on BASELINE config 2 (5 Mbp x 100x, seed 2): the same records written both ways, `polish` of each.
Writes the JSON (default profiles/bam_bench.json) with the GPU name and power limit.
usage: python tools/bam_bench.py [out.json] [contig_len] [depth]

Reported per input format: file sizes; pp_polish_files wall time (best of 4, page cache warm); the load through pp_tok_add_files
(h2d_ms: for BAM read + inflate + record walk + PCIe, for SAM read + PCIe; device_ms: the decode / tokeniser kernels, CUDA events);
pp_polish_resident on the loaded dataset; and, from the log of a verbose pp_polish_files run (best of 4), the load split per file:
for BAM read, inflate, record walk, image to HBM and the kernels (k_bam_parse, the scans, k_bam_emit, k_tok_heads, k_tok_groups);
for SAM text to HBM and the tokeniser kernels; then the polish kernels of the GPU job."""
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as g  # noqa: E402

g.build()
import polypolish_b200 as pp  # noqa: E402
from polypolish_b200 import api  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "bam_bench.json")
clen = int(sys.argv[2]) if len(sys.argv) > 2 else 5_000_000
depth = float(sys.argv[3]) if len(sys.argv) > 3 else 100.0


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        n, p = [x.strip() for x in q.stdout.strip().split(",")]
        return dict(gpu=n, power_limit=p)
    except Exception as e:  # noqa: BLE001
        return dict(gpu="unknown", power_limit="unknown", error=str(e))


def best_of(f, k=4):
    best = None
    for _ in range(k):
        t0 = time.perf_counter()
        r = f()
        ms = (time.perf_counter() - t0) * 1e3
        best = ms if best is None else min(best, ms)
    return best, r


def verbose_split(ctx, fa, files):
    """One verbose pp_polish_files run with the library's stderr captured: the per-file load lines and the GPU job line as numbers."""
    with tempfile.TemporaryFile() as tf:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(tf.fileno(), 2)
        try:
            ctx.polish_files(fa, files, verbose=True)
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        tf.seek(0)
        log = tf.read().decode("utf-8", "replace")
    files_out = []
    for ln in log.splitlines():
        m = re.match(r"BAM decoder .*: ([\d,]+) records, read ([\d.]+) ms, inflate ([\d.]+) ms, record walk ([\d.]+) ms, "
                     r"image to HBM ([\d.]+) ms, (\d+) kernels ([\d.]+) ms", ln)
        if m:
            files_out.append(dict(records=int(m.group(1).replace(",", "")), read_ms=float(m.group(2)), inflate_ms=float(m.group(3)),
                                  walk_ms=float(m.group(4)), h2d_ms=float(m.group(5)), kernels=int(m.group(6)), kernels_ms=float(m.group(7))))
        m = re.match(r"SAM tokeniser .*: ([\d,]+) lines, text to HBM ([\d.]+) ms, (\d+) kernels ([\d.]+) ms", ln)
        if m:
            files_out.append(dict(lines=int(m.group(1).replace(",", "")), h2d_ms=float(m.group(2)), kernels=int(m.group(3)),
                                  kernels_ms=float(m.group(4))))
    m = re.search(r"GPU job 0: .* device path ([\d.]+) ms", log)
    return dict(files=files_out, polish_device_ms=float(m.group(1)) if m else None)


base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 6 << 30 else None
d = tempfile.mkdtemp(prefix="pp_bambench_", dir=base)
out = dict(config="BASELINE config 2", contig_len=clen, depth=depth, **gpu_info())
try:
    syn = api.Synth(seed=2, contig_len=clen, depth=depth)
    fa, sams = syn.write(d)
    os.makedirs(os.path.join(d, "b"))
    t0 = time.perf_counter()
    _, bams = syn.write(os.path.join(d, "b"), bam=True)
    out["write_bam_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
    fasta = pp.load_fasta(fa)
    with pp.Context(0) as ctx:
        results = {}
        for kind, files in (("sam", sams), ("bam", bams)):
            r = dict(bytes=[os.path.getsize(x) for x in files])
            r["polish_files_ms"], fasta_out = best_of(lambda: ctx.polish_files(fa, files))
            results[kind + "_fasta"] = fasta_out
            loads = []
            for _ in range(4):
                t0 = time.perf_counter()
                rc, st = ctx.tokenise(fasta, files)
                wall = (time.perf_counter() - t0) * 1e3
                assert rc == 0, rc
                loads.append(dict(wall_ms=round(wall, 2), h2d_ms=[round(s["h2d_ms"], 2) for s in st],
                                  device_ms=[round(s["device_ms"], 3) for s in st], launches=[s["launches"] for s in st],
                                  records=[s["lines"] for s in st], alignments=[s["alignments"] for s in st]))
            r["load"] = min(loads, key=lambda x: x["wall_ms"])
            splits = [verbose_split(ctx, fa, files) for _ in range(4)]
            r["split"] = min(splits, key=lambda x: sum(f["h2d_ms"] + f.get("read_ms", 0) + f.get("inflate_ms", 0) + f.get("walk_ms", 0)
                                                        for f in x["files"]))
            r["polish_resident_ms"], _ = best_of(lambda: ctx.polish_resident(fetch=False))
            r["polish_files_ms"] = round(r["polish_files_ms"], 2)
            r["polish_resident_ms"] = round(r["polish_resident_ms"], 2)
            out[kind] = r
        out["same_fasta"] = results["sam_fasta"] == results["bam_fasta"]
    out["not_measured"] = ("the k_bam_* kernels are not timed apart from the scans and group kernels they share with the SAM path "
                           "(kernels_ms covers all of them); GPU inflate does not exist yet")
finally:
    shutil.rmtree(d, ignore_errors=True)
os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
text = json.dumps(out, indent=1)
print(text)
with open(out_path, "w") as fh:
    fh.write(text + "\n")
