"""Builds and binds tests/emu/emu_polish.cpp: the polish kernels (polypolish_b200/csrc/polish_dev.cuh) compiled for the CPU
against a small CUDA-emulation shim.  TEST INFRASTRUCTURE ONLY (logic checks without a GPU); never used by the product."""
import ctypes as C
import os
import subprocess

import numpy as np

from polypolish_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "emu", "emu_polish.cpp")
LIB = os.path.join(ROOT, "build", "libemu_polish.so")
DEPS = [SRC, os.path.join(ROOT, "tests", "emu", "cuda_emu.h"), os.path.join(ROOT, "polypolish_b200", "csrc", "polish_dev.cuh"),
        os.path.join(ROOT, "polypolish_b200", "csrc", "nib_utils.h"), os.path.join(ROOT, "include", "pp_abi.h")]


def build():
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in DEPS):
        tmp = "%s.%d.tmp" % (LIB, os.getpid())           # several test workers may build at once: compile aside, rename atomically
        subprocess.check_call(["g++", "-std=c++20", "-O2", "-g", "-shared", "-fPIC", "-pthread", "-Wall", "-Wno-unknown-pragmas", "-Wno-unused-function",
                               "-Wno-unused-variable", "-ffp-contract=off", "-I", os.path.join(ROOT, "tests", "emu"), SRC, "-o", tmp])
        os.replace(tmp, LIB)
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.emu_polish.argtypes = [C.POINTER(api.Contigs), C.POINTER(api.Alignments), C.POINTER(api.PolishParams), C.POINTER(api.PolishResult),
                                    C.c_int, C.POINTER(C.c_ulonglong)]
        _lib.emu_polish_ex.argtypes = [C.POINTER(api.Contigs), C.POINTER(api.Alignments), C.POINTER(api.PolishParams),
                                       C.POINTER(api.PolishResult), C.c_int, C.c_ulonglong, C.c_ulonglong, C.POINTER(EmuReport),
                                       C.POINTER(C.c_ulonglong)]
        _lib.emu_make_sig.restype = C.c_ulonglong
        _lib.emu_make_sig.argtypes = [C.c_int, C.c_char_p, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.c_uint32]
        _lib.emu_sig_exact.argtypes = [C.c_int, C.c_ulonglong]
        _lib.emu_allele_equal.argtypes = [C.c_int, C.c_char_p] + [C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.c_uint32] * 2
    return _lib


class EmuReport(C.Structure):
    """What one emulated call saw (tests/emu/emu_polish.cpp)."""
    _fields_ = [("first_rc", C.c_int), ("flags", C.c_uint), ("node_count", C.c_uint), ("global_k", C.c_uint), ("out_len", C.c_ulonglong),
                ("node_cap", C.c_ulonglong), ("out_cap", C.c_ulonglong), ("guards_ok", C.c_int)]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


# DevStatus.flags (polish_dev.cuh)
FL_NODE_OVF, FL_OUT_OVF, FL_BIGGROUP = 1, 8, 16
BIGGROUP_RC = 100          # emu_polish_ex's first pass ends with this when a read group was too large for k_goodk's scan

ERR_TEXT = {1: "query name in SAM but not in assembly", 2: "CIGAR string does not match read sequence", 3: "unexpected character",
            4: "alignment extends past the end of its reference sequence", 5: "no alignments for read contain sequence"}


def polish(fasta, packed, grid_tiles=2, node_cap=0, out_cap=0, **opts):
    """The emulated kernels on a loaded assembly + packed alignments: dict like Context.polish_packed (plus `report`, what the call
    saw: EmuReport.as_dict()), or dict(error=..., error_aln=...).  node_cap / out_cap: the node pool and output buffer the kernels get
    (0 = the emulator's default); an overflow returns dict(overflow=report)."""
    prm = api._params(**opts)
    n = fasta.view.n_contigs
    G = int(fasta.off[-1])
    cap = max(G + G // 4 + (1 << 20), out_cap)
    keep = dict(off=np.zeros(n + 1, np.uint64), bases=np.zeros(cap, np.uint8), changed=np.zeros(n, np.uint64), zero=np.zeros(n, np.uint64),
                tdepth=np.zeros(n, np.float64))
    res = api.PolishResult()
    res.out_off, res.out_bases, res.out_cap = keep["off"].ctypes.data, keep["bases"].ctypes.data, cap
    res.changed, res.zero_depth, res.total_depth = keep["changed"].ctypes.data, keep["zero"].ctypes.data, keep["tdepth"].ctypes.data
    err = C.c_ulonglong()
    rep = EmuReport()
    rc = lib().emu_polish_ex(C.byref(fasta.view), C.byref(packed.view), C.byref(prm), C.byref(res), grid_tiles, node_cap, out_cap,
                             C.byref(rep), C.byref(err))
    if rc == api.PP_ERR_INPUT:
        return dict(error=ERR_TEXT.get(err.value & 0xFF, "?"), error_aln=err.value >> 8, report=rep.as_dict())
    if rc == api.PP_ERR_NOMEM:
        return dict(overflow=rep.as_dict())
    assert rc == 0, rc
    off = keep["off"]
    return dict(sequences=[keep["bases"][int(off[i]):int(off[i + 1])].tobytes() for i in range(n)], changed=keep["changed"].tolist(),
                zero_depth=keep["zero"].tolist(), total_depth=keep["tdepth"].tolist(), n_aln_used=res.n_aln_used, report=rep.as_dict())


def fasta_bytes(fasta, seqs):
    return b"".join(b">" + fasta.names[i].encode() + ((b" " + fasta.descriptions[i].encode()) if fasta.descriptions[i] else b"") +
                    b" polypolish\n" + seqs[i] + b"\n" for i in range(len(seqs)))
