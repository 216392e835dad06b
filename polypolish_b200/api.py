"""ctypes mirror of include/pp_abi.h.

Names follow the reference's command surface (main.rs:44-109): `polish(...)` and `filter_sams(...)` take the same
options with the same defaults and raise PolypolishError with the reference's error text.
"""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PP_OK, PP_ERR_CUDA, PP_ERR_ARG, PP_ERR_INPUT, PP_ERR_NOMEM, PP_ERR_IO = 0, -1, -2, -3, -4, -5
N_STAGES = 8
STAGES = ["reset", "classify", "goodk", "tile", "compact", "unused", "h2d", "d2h"]


class PolypolishError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[{code}] {msg}")
        self.code = code
        self.msg = msg


def lib_path():
    """The in-tree library; POLYPOLISH_LIB selects another build of it (kernel experiments)."""
    return os.environ.get("POLYPOLISH_LIB") or os.path.join(ROOT, "build", "libpolypolish_b200.so")


class Alignments(C.Structure):
    _fields_ = [("n_aln", C.c_uint64), ("n_reads", C.c_uint64),
                ("contig", C.c_void_p), ("ref_start", C.c_void_p), ("read_id", C.c_void_p), ("seq_off", C.c_void_p),
                ("seq_len", C.c_void_p), ("cigar_off", C.c_void_p), ("n_cigar", C.c_void_p), ("nm", C.c_void_p),
                ("flags", C.c_void_p), ("n_cigar_ops", C.c_uint64), ("cigar_ops", C.c_void_p),
                ("seq_bits", C.c_uint32), ("seq_pool_bytes", C.c_uint64), ("seq_pool", C.c_void_p),
                ("esc_pool_bytes", C.c_uint64), ("esc_pool", C.c_void_p)]


class Contigs(C.Structure):
    _fields_ = [("n_contigs", C.c_uint32), ("off", C.c_void_p), ("bases", C.c_void_p)]


class PolishParams(C.Structure):
    _fields_ = [("fraction_invalid", C.c_double), ("fraction_valid", C.c_double), ("max_errors", C.c_uint32),
                ("min_depth", C.c_uint32), ("careful", C.c_int32)]


class Timing(C.Structure):
    _fields_ = [("total_ms", C.c_float), ("stage_ms", C.c_float * N_STAGES), ("launches", C.c_uint32),
                ("reserved", C.c_uint32)]

    def as_dict(self):
        d = {"total_ms": self.total_ms, "launches": self.launches}
        d.update({STAGES[i] + "_ms": self.stage_ms[i] for i in range(N_STAGES)})
        return d


class PolishResult(C.Structure):
    _fields_ = [("out_off", C.c_void_p), ("out_bases", C.c_void_p), ("out_cap", C.c_uint64), ("changed", C.c_void_p),
                ("zero_depth", C.c_void_p), ("total_depth", C.c_void_p), ("out_len", C.c_uint64), ("n_aln_used", C.c_uint64),
                ("error_aln", C.c_int64), ("timing", Timing)]


class FilterMate(C.Structure):
    _fields_ = [("n", C.c_uint64), ("name_id", C.c_void_p), ("contig", C.c_void_p), ("ref_start", C.c_void_p),
                ("ref_end", C.c_void_p), ("flags", C.c_void_p)]


class FilterParams(C.Structure):
    _fields_ = [("orientation", C.c_int32), ("low_pct", C.c_double), ("high_pct", C.c_double),
                ("n_names", C.c_uint64)]


class FilterResult(C.Structure):
    _fields_ = [("pass1", C.c_void_p), ("pass2", C.c_void_p), ("low", C.c_uint32), ("high", C.c_uint32),
                ("orientation", C.c_int32), ("pairs", C.c_uint64 * 4), ("n_pass", C.c_uint64), ("timing", Timing)]


class TokStats(C.Structure):
    _fields_ = [("lines", C.c_uint64), ("alignments", C.c_uint64), ("reads", C.c_uint64), ("h2d_ms", C.c_float),
                ("device_ms", C.c_float), ("launches", C.c_uint32), ("h2d_bytes", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


PP_TOK_HOST = 1
PP_TOK_NEED8 = 2

_lib = None


def lib():
    """Loads the CUDA library.  Fails loudly: there is no CPU path behind this package."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise PolypolishError(PP_ERR_CUDA, f"{p} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                           "(nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(p)
    L.pp_version.restype = C.c_char_p
    L.pp_last_error.restype = C.c_char_p
    L.pp_last_error.argtypes = [C.c_void_p]
    L.pp_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.pp_destroy.argtypes = [C.c_void_p]
    L.pp_host_alloc.restype = C.c_void_p
    L.pp_host_alloc.argtypes = [C.c_size_t]
    L.pp_host_free.argtypes = [C.c_void_p]
    L.pp_polish.argtypes = [C.c_void_p, C.POINTER(Contigs), C.POINTER(Alignments), C.POINTER(PolishParams),
                            C.POINTER(PolishResult)]
    L.pp_dataset_upload.argtypes = [C.c_void_p, C.POINTER(Contigs), C.POINTER(Alignments)]
    L.pp_polish_resident.argtypes = [C.c_void_p, C.POINTER(PolishParams), C.POINTER(PolishResult)]
    L.pp_fasta_load.restype = C.c_void_p
    L.pp_fasta_load.argtypes = [C.c_char_p, C.c_char_p, C.c_size_t]
    L.pp_fasta_free.argtypes = [C.c_void_p]
    L.pp_fasta_view.argtypes = [C.c_void_p, C.POINTER(Contigs)]
    L.pp_fasta_name.restype = C.c_char_p
    L.pp_fasta_name.argtypes = [C.c_void_p, C.c_uint32]
    L.pp_fasta_description.restype = C.c_char_p
    L.pp_fasta_description.argtypes = [C.c_void_p, C.c_uint32]
    L.pp_pack_create.restype = C.c_void_p
    L.pp_pack_create.argtypes = [C.c_void_p, C.c_int]
    L.pp_pack_free.argtypes = [C.c_void_p]
    L.pp_pack_add_sam_file.argtypes = [C.c_void_p, C.c_char_p]
    L.pp_pack_add_sam_text.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, C.c_char_p]
    L.pp_pack_finish.argtypes = [C.c_void_p, C.POINTER(Alignments)]
    L.pp_pack_error.restype = C.c_char_p
    L.pp_pack_error.argtypes = [C.c_void_p]
    L.pp_pack_unknown_ref.restype = C.c_char_p
    L.pp_pack_unknown_ref.argtypes = [C.c_void_p, C.c_uint64]
    L.pp_pack_read_name.restype = C.c_char_p
    L.pp_pack_read_name.argtypes = [C.c_void_p, C.c_uint64]
    L.pp_pack_file_stats.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.pp_polish_files.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_char_p), C.c_int, C.POINTER(PolishParams),
                                  C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_int]
    L.pp_free.argtypes = [C.c_void_p]
    L.pp_tok_begin.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.pp_tok_add_text.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, C.POINTER(TokStats)]
    L.pp_tok_add_file.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(TokStats)]
    L.pp_tok_finish.argtypes = [C.c_void_p]
    L.pp_tok_add_files.argtypes = [C.c_void_p, C.POINTER(C.c_char_p), C.c_int, C.POINTER(TokStats)]
    L.pp_tok_prefetch.argtypes = [C.c_void_p, C.c_char_p]
    L.pp_tok_expect.argtypes = [C.c_void_p, C.c_uint64]
    L.pp_set_parser.argtypes = [C.c_void_p, C.c_int]
    L.pp_get_parser.argtypes = [C.c_void_p]
    L.pp_tok_set_readers.argtypes = [C.c_void_p, C.c_int]
    L.pp_tok_set_strip_qual.argtypes = [C.c_void_p, C.c_int]
    L.pp_dataset_sizes.argtypes = [C.c_void_p, C.POINTER(Alignments)]
    L.pp_dataset_download.argtypes = [C.c_void_p, C.POINTER(Alignments)]
    if hasattr(L, "pp_filter"):
        L.pp_filter.argtypes = [C.c_void_p, C.POINTER(FilterMate), C.POINTER(FilterMate), C.POINTER(FilterParams),
                                C.POINTER(FilterResult)]
    if hasattr(L, "pp_filter_files"):
        L.pp_filter_files.argtypes = [C.c_void_p] + [C.c_char_p] * 5 + [C.c_double, C.c_double, C.c_int]
    _lib = L
    return L


def _params(fraction_invalid=0.2, fraction_valid=0.5, max_errors=10, min_depth=5, careful=False):
    return PolishParams(fraction_invalid, fraction_valid, max_errors, min_depth, int(bool(careful)))


class Fasta:
    """misc::load_fasta (misc.rs:38-167) result, host side."""

    def __init__(self, path):
        L = lib()
        err = C.create_string_buffer(1024)
        self.h = L.pp_fasta_load(str(path).encode(), err, 1024)
        if not self.h:
            raise PolypolishError(PP_ERR_INPUT, err.value.decode())
        self.view = Contigs()
        L.pp_fasta_view(self.h, C.byref(self.view))
        n = self.view.n_contigs
        self.names = [L.pp_fasta_name(self.h, i).decode() for i in range(n)]
        self.descriptions = [L.pp_fasta_description(self.h, i).decode() for i in range(n)]
        self.off = np.ctypeslib.as_array(C.cast(self.view.off, C.POINTER(C.c_uint64)), shape=(n + 1,)).copy()

    def sequence(self, i):
        return C.string_at(self.view.bases + int(self.off[i]), int(self.off[i + 1] - self.off[i]))

    def records(self):
        return [(self.names[i], self.descriptions[i], self.sequence(i).decode("latin-1")) for i in range(len(self.names))]

    def close(self):
        if self.h:
            lib().pp_fasta_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def load_fasta(path):
    return Fasta(path)


class Packed:
    """SAM text -> pp_alignments (host side; sam_pack.cpp)."""

    def __init__(self, fasta, careful=False):
        self.fasta = fasta
        self.h = lib().pp_pack_create(fasta.h, int(bool(careful)))
        self.view = None

    def _check(self, rc):
        if rc != PP_OK:
            raise PolypolishError(rc, lib().pp_pack_error(self.h).decode("utf-8", "replace"))

    def set_threads(self, n_threads, min_chunk_bytes=8 << 20):
        L = lib()
        L.pp_pack_set_threads.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64]
        L.pp_pack_set_threads(self.h, n_threads, min_chunk_bytes)

    def add_file(self, path):
        self._check(lib().pp_pack_add_sam_file(self.h, str(path).encode()))

    def add_text(self, text, name="<memory>"):
        if isinstance(text, str):
            text = text.encode("latin-1")
        self._check(lib().pp_pack_add_sam_text(self.h, text, len(text), name.encode()))

    def finish(self):
        self.view = Alignments()
        self._check(lib().pp_pack_finish(self.h, C.byref(self.view)))
        return self.view

    def arrays(self):
        """numpy views of the SoA arrays (valid while this object lives)."""
        v = self.view
        n = v.n_aln

        def arr(ptr, ct, cnt):
            if cnt == 0:
                return np.zeros(0, dtype=ct)
            return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), shape=(cnt,))
        return dict(contig=arr(v.contig, C.c_uint32, n), ref_start=arr(v.ref_start, C.c_uint32, n),
                    read_id=arr(v.read_id, C.c_uint32, n), seq_off=arr(v.seq_off, C.c_uint32, n),
                    seq_len=arr(v.seq_len, C.c_uint16, n), cigar_off=arr(v.cigar_off, C.c_uint32, n),
                    n_cigar=arr(v.n_cigar, C.c_uint16, n), nm=arr(v.nm, C.c_uint32, n), flags=arr(v.flags, C.c_uint8, n),
                    cigar_ops=arr(v.cigar_ops, C.c_uint32, v.n_cigar_ops), seq_pool=arr(v.seq_pool, C.c_uint8, v.seq_pool_bytes),
                    seq_bits=v.seq_bits, n_reads=v.n_reads)

    def read_name(self, aln):
        return lib().pp_pack_read_name(self.h, aln).decode()

    def close(self):
        if self.h:
            lib().pp_pack_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def pack_sams(fasta, sams, careful=False):
    p = Packed(fasta, careful)
    for s in sams:
        p.add_file(s)
    p.finish()
    return p


class Context:
    """One pp_ctx = one GPU."""

    def __init__(self, device=0):
        L = lib()
        h = C.c_void_p()
        rc = L.pp_create(device, C.byref(h))
        if rc != PP_OK:
            raise PolypolishError(rc, "pp_create failed: no usable sm_100 CUDA device (there is no CPU fallback)")
        self.h = h

    def _err(self, rc):
        return PolypolishError(rc, lib().pp_last_error(self.h).decode("utf-8", "replace"))

    def close(self):
        if self.h:
            lib().pp_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- packed level -------------------------------------------------------------------------------------
    def _result(self, n_contigs, cap):
        res = PolishResult()
        keep = dict(off=np.zeros(n_contigs + 1, dtype=np.uint64), bases=np.zeros(max(1, cap), dtype=np.uint8),
                    changed=np.zeros(n_contigs, dtype=np.uint64), zero=np.zeros(n_contigs, dtype=np.uint64),
                    tdepth=np.zeros(n_contigs, dtype=np.float64))
        res.total_depth = keep["tdepth"].ctypes.data
        res.out_off = keep["off"].ctypes.data
        res.out_bases = keep["bases"].ctypes.data
        res.out_cap = cap
        res.changed = keep["changed"].ctypes.data
        res.zero_depth = keep["zero"].ctypes.data
        return res, keep

    def _finish(self, res, keep, n_contigs):
        off = keep["off"]
        seqs = [keep["bases"][int(off[i]):int(off[i + 1])].tobytes() for i in range(n_contigs)]
        return dict(sequences=seqs, changed=keep["changed"].tolist(), zero_depth=keep["zero"].tolist(),
                    total_depth=keep["tdepth"].tolist(), n_aln_used=res.n_aln_used, out_len=res.out_len, timing=res.timing.as_dict())

    def pinned_result(self, n_contigs, cap):
        """Caller-owned result buffers in pinned host memory (pp_host_alloc), reusable across pp_polish calls."""
        L = lib()
        nbytes = [8 * (n_contigs + 1), max(1, cap), 8 * n_contigs, 8 * n_contigs]
        ptrs = [L.pp_host_alloc(n) for n in nbytes]
        if not all(ptrs):
            raise PolypolishError(PP_ERR_NOMEM, "pp_host_alloc failed")
        keep = dict(off=np.ctypeslib.as_array(C.cast(ptrs[0], C.POINTER(C.c_uint64)), shape=(n_contigs + 1,)),
                    bases=np.ctypeslib.as_array(C.cast(ptrs[1], C.POINTER(C.c_uint8)), shape=(max(1, cap),)),
                    changed=np.ctypeslib.as_array(C.cast(ptrs[2], C.POINTER(C.c_uint64)), shape=(n_contigs,)),
                    zero=np.ctypeslib.as_array(C.cast(ptrs[3], C.POINTER(C.c_uint64)), shape=(n_contigs,)), _pinned=ptrs)
        res = PolishResult()
        res.out_off, res.out_bases, res.out_cap, res.changed, res.zero_depth = ptrs[0], ptrs[1], cap, ptrs[2], ptrs[3]
        return res, keep

    def free_pinned_result(self, keep):
        for p in keep.pop("_pinned", []):
            lib().pp_host_free(p)

    def polish_packed(self, contigs, alns, into=None, **opts):
        """pp_polish: host SoA in, host bases out (H2D / D2H inside).  `into` = (res, keep) from pinned_result(): the
        result lands in those buffers and only the statistics are returned (no per-call allocation)."""
        prm = _params(**opts)
        if into is not None:
            res, keep = into
            rc = lib().pp_polish(self.h, C.byref(contigs), C.byref(alns), C.byref(prm), C.byref(res))
            if rc != PP_OK:
                raise self._err(rc)
            return dict(n_aln_used=res.n_aln_used, out_len=res.out_len, timing=res.timing.as_dict())
        G = int(np.ctypeslib.as_array(C.cast(contigs.off, C.POINTER(C.c_uint64)), shape=(contigs.n_contigs + 1,))[-1])
        cap = G + (1 << 20)
        for _ in range(2):
            res, keep = self._result(contigs.n_contigs, cap)
            rc = lib().pp_polish(self.h, C.byref(contigs), C.byref(alns), C.byref(prm), C.byref(res))
            if rc == PP_ERR_ARG and res.out_len > cap:
                cap = int(res.out_len)
                continue
            break
        if rc != PP_OK:
            e = self._err(rc)
            e.error_aln = res.error_aln
            raise e
        return self._finish(res, keep, contigs.n_contigs)

    def upload(self, contigs, alns):
        rc = lib().pp_dataset_upload(self.h, C.byref(contigs), C.byref(alns))
        if rc != PP_OK:
            raise self._err(rc)
        self._nc = contigs.n_contigs
        self._G = int(np.ctypeslib.as_array(C.cast(contigs.off, C.POINTER(C.c_uint64)), shape=(contigs.n_contigs + 1,))[-1])

    def polish_resident(self, fetch=True, **opts):
        prm = _params(**opts)
        cap = self._G + (1 << 20) if fetch else 0
        for _ in range(2):
            if fetch:
                res, keep = self._result(self._nc, cap)
            else:
                res, keep = PolishResult(), None
            rc = lib().pp_polish_resident(self.h, C.byref(prm), C.byref(res))
            if fetch and rc == PP_ERR_ARG and res.out_len > cap:
                cap = int(res.out_len)
                continue
            break
        if rc != PP_OK:
            raise self._err(rc)
        if not fetch:
            return dict(n_aln_used=res.n_aln_used, out_len=res.out_len, timing=res.timing.as_dict())
        return self._finish(res, keep, self._nc)

    # ---- device SAM tokeniser (tok_kernels.cu) ------------------------------------------------------------------
    def tokenise(self, fasta, sources, careful=False, seq_bits=4):
        """SAM texts (bytes) or files (paths) -> resident dataset, parsed on the device.  Returns (rc, [stats]) where rc is
        PP_OK, PP_TOK_HOST or PP_TOK_NEED8; errors raise."""
        L = lib()
        rc = L.pp_tok_begin(self.h, fasta.h, int(bool(careful)), seq_bits)
        if rc != PP_OK:
            raise self._err(rc)
        stats = []
        if sources and not any(isinstance(x, (bytes, bytearray)) for x in sources):
            # files: the pipelined call (file i+1 streams in while file i is tokenised)
            L.pp_tok_expect(self.h, sum(os.path.getsize(str(x)) for x in sources if os.path.exists(str(x))))
            arr = (C.c_char_p * len(sources))(*[str(x).encode() for x in sources])
            sts = (TokStats * len(sources))()
            rc = L.pp_tok_add_files(self.h, arr, len(sources), sts)
            if rc < 0:
                raise self._err(rc)
            stats = [st.as_dict() for st in sts]
            if rc != PP_OK:
                return rc, stats
            sources = []
        for src in sources:
            st = TokStats()
            if isinstance(src, (bytes, bytearray)):
                rc = L.pp_tok_add_text(self.h, bytes(src), len(src), C.byref(st))
            else:
                rc = L.pp_tok_add_file(self.h, str(src).encode(), C.byref(st))
            if rc < 0:
                raise self._err(rc)
            stats.append(st.as_dict())
            if rc != PP_OK:
                return rc, stats
        rc = L.pp_tok_finish(self.h)
        if rc != PP_OK:
            raise self._err(rc)
        self._nc = fasta.view.n_contigs
        self._G = int(fasta.off[-1])
        return PP_OK, stats

    def dataset_arrays(self):
        """The resident dataset copied back to the host (same keys as Packed.arrays())."""
        L = lib()
        v = Alignments()
        rc = L.pp_dataset_sizes(self.h, C.byref(v))
        if rc != PP_OK:
            raise self._err(rc)
        n = v.n_aln
        a = dict(contig=np.zeros(n, np.uint32), ref_start=np.zeros(n, np.uint32), read_id=np.zeros(n, np.uint32),
                 seq_off=np.zeros(n, np.uint32), seq_len=np.zeros(n, np.uint16), cigar_off=np.zeros(n, np.uint32),
                 n_cigar=np.zeros(n, np.uint16), nm=np.zeros(n, np.uint32), flags=np.zeros(n, np.uint8),
                 cigar_ops=np.zeros(v.n_cigar_ops, np.uint32), seq_pool=np.zeros(v.seq_pool_bytes, np.uint8))
        for k, arr in a.items():
            setattr(v, k, arr.ctypes.data)
        rc = L.pp_dataset_download(self.h, C.byref(v))
        if rc != PP_OK:
            raise self._err(rc)
        a["seq_bits"] = v.seq_bits
        a["n_reads"] = v.n_reads
        return a

    def set_readers(self, n):
        """Host threads streaming a SAM file into HBM (0 = automatic)."""
        lib().pp_tok_set_readers(self.h, int(n))

    def set_strip_qual(self, on):
        """Whether SAM files are uploaded without their QUAL column (default off; polish never reads it, but the stripping is host-bound)."""
        lib().pp_tok_set_strip_qual(self.h, int(bool(on)))

    def set_parser(self, mode):
        """0: pp_polish_files parses SAM on the device (default); 1: on the host."""
        lib().pp_set_parser(self.h, int(mode))

    # ---- file level (what the CLI does) ----------------------------------------------------------------------
    def polish_files(self, assembly, sams, debug=None, verbose=False, **opts):
        prm = _params(**opts)
        arr = (C.c_char_p * max(1, len(sams)))(*[str(s).encode() for s in sams])
        out = C.c_void_p()
        n = C.c_uint64()
        rc = lib().pp_polish_files(self.h, str(assembly).encode(), arr, len(sams), C.byref(prm),
                                   str(debug).encode() if debug else None, C.byref(out), C.byref(n), int(verbose))
        if rc != PP_OK:
            raise self._err(rc)
        data = C.string_at(out, n.value)
        lib().pp_free(out)
        return data

    def filter_polish_files(self, assembly, in1, in2, out1=None, out2=None, orientation="auto", low=0.1, high=99.9, verbose=False, **opts):
        """pp_filter_polish_files: `filter` then `polish` in one call (the filtered SAM files are written only when named)."""
        L = lib()
        L.pp_filter_polish_files.argtypes = [C.c_void_p] + [C.c_char_p] * 6 + [C.c_double, C.c_double, C.POINTER(PolishParams),
                                                                              C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_int]
        prm = _params(**opts)
        out, n = C.c_void_p(), C.c_uint64()
        rc = L.pp_filter_polish_files(self.h, str(assembly).encode(), str(in1).encode(), str(in2).encode(),
                                      str(out1).encode() if out1 else None, str(out2).encode() if out2 else None, orientation.encode(),
                                      low, high, C.byref(prm), C.byref(out), C.byref(n), int(verbose))
        if rc != PP_OK:
            raise self._err(rc)
        data = C.string_at(out, n.value)
        L.pp_free(out)
        return data

    def filter_files(self, in1, in2, out1, out2, orientation="auto", low=0.1, high=99.9, verbose=False):
        rc = lib().pp_filter_files(self.h, str(in1).encode(), str(in2).encode(), str(out1).encode(), str(out2).encode(),
                                   orientation.encode(), low, high, int(verbose))
        if rc != PP_OK:
            raise self._err(rc)


def polish_files(assembly, sams, device=0, **kw):
    with Context(device) as ctx:
        return ctx.polish_files(assembly, sams, **kw)


def polish(assembly, sam, debug=None, fraction_invalid=0.2, fraction_valid=0.5, max_errors=10, min_depth=5,
           careful=False, device=0):
    """`polypolish polish` (main.rs:78-108, polish.rs:26-38): returns the bytes the reference prints to stdout."""
    return polish_files(assembly, list(sam), device=device, debug=debug, fraction_invalid=fraction_invalid,
                        fraction_valid=fraction_valid, max_errors=max_errors, min_depth=min_depth, careful=careful)


def filter_sams(in1, in2, out1, out2, orientation="auto", low=0.1, high=99.9, device=0):
    """`polypolish filter` (main.rs:47-75, filter.rs:26-37)."""
    with Context(device) as ctx:
        ctx.filter_files(in1, in2, out1, out2, orientation, low, high)


# ---- synthetic inputs (measurement / test support; csrc/synth.cpp) -------------------------------------------
class SynthParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("n_contigs", C.c_uint32), ("read_len", C.c_uint32), ("contig_len", C.c_uint64),
                ("depth", C.c_double), ("insert_mean", C.c_double), ("insert_sd", C.c_double),
                ("draft_error_rate", C.c_double), ("seq_sub_rate", C.c_double), ("seq_indel_rate", C.c_double),
                ("repeat_fraction", C.c_double), ("clip_rate", C.c_double), ("highnm_rate", C.c_double),
                ("unaligned_rate", C.c_double)]


class Synth:
    """Deterministic synthetic contigs + bwa-mem -a style paired SAM (SURVEY.md §8d)."""

    def __init__(self, seed=1, n_contigs=1, contig_len=50_000, depth=100.0, read_len=150, insert_mean=400.0,
                 insert_sd=40.0, draft_error_rate=1e-4, seq_sub_rate=2e-3, seq_indel_rate=1e-4, repeat_fraction=0.03,
                 clip_rate=0.005, highnm_rate=0.005, unaligned_rate=0.005, cross_contig=0.0):
        L = lib()
        L.pp_synth_create.restype = C.c_void_p
        L.pp_synth_create.argtypes = [C.POINTER(SynthParams)]
        L.pp_synth_free.argtypes = [C.c_void_p]
        L.pp_synth_total_bp.restype = C.c_uint64
        L.pp_synth_total_bp.argtypes = [C.c_void_p]
        L.pp_synth_n_pairs.restype = C.c_uint64
        L.pp_synth_n_pairs.argtypes = [C.c_void_p]
        L.pp_synth_write_fasta.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.pp_synth_write_sam.argtypes = [C.c_void_p, C.c_int, C.c_char_p]
        L.pp_synth_fasta.restype = C.c_void_p
        L.pp_synth_fasta.argtypes = [C.c_void_p]
        L.pp_synth_feed_pack.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        prm = SynthParams(seed, n_contigs, read_len, contig_len, depth, insert_mean, insert_sd, draft_error_rate,
                          seq_sub_rate, seq_indel_rate, repeat_fraction, clip_rate, highnm_rate, unaligned_rate)
        L.pp_synth_create_shared.restype = C.c_void_p
        L.pp_synth_create_shared.argtypes = [C.POINTER(SynthParams), C.c_double]
        self.h = L.pp_synth_create_shared(C.byref(prm), float(cross_contig)) if cross_contig else L.pp_synth_create(C.byref(prm))
        if not self.h:
            raise PolypolishError(PP_ERR_ARG, "pp_synth_create: bad parameters")
        self.total_bp = L.pp_synth_total_bp(self.h)
        self.n_pairs = L.pp_synth_n_pairs(self.h)

    def set_shard_filter(self, n_shards, shard, shard_of_contig=None):
        """Cross-contig data sets: emit only the reads with a record on a contig of `shard` (n_shards = 0: everything again)."""
        L = lib()
        L.pp_synth_set_shard_filter.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]
        arr = None
        if shard_of_contig is not None:
            arr = (C.c_uint32 * len(shard_of_contig))(*[int(x) for x in shard_of_contig])
        rc = L.pp_synth_set_shard_filter(self.h, n_shards, shard, arr)
        if rc != PP_OK:
            raise PolypolishError(rc, "pp_synth_set_shard_filter: needs a cross-contig data set and shard < n_shards")

    def set_threads(self, n_threads):
        """Generator threads (cross-contig data sets only; same bytes whatever the count).  0 = one per hardware thread."""
        L = lib()
        L.pp_synth_set_threads.argtypes = [C.c_void_p, C.c_uint32]
        L.pp_synth_set_threads(self.h, int(n_threads))

    def write(self, directory, bam=False):
        """draft FASTA + one SAM (bam=True: BAM, the same records) per mate; returns (fasta, [file1, file2])."""
        d = str(directory)
        L = lib()
        L.pp_synth_write_bam.argtypes = [C.c_void_p, C.c_int, C.c_char_p]
        ext, wr = (".bam", L.pp_synth_write_bam) if bam else (".sam", L.pp_synth_write_sam)
        fa, s1, s2 = os.path.join(d, "draft.fasta"), os.path.join(d, "reads_1" + ext), os.path.join(d, "reads_2" + ext)
        for rc in (L.pp_synth_write_fasta(self.h, fa.encode(), 0), wr(self.h, 1, s1.encode()), wr(self.h, 2, s2.encode())):
            if rc != PP_OK:
                raise PolypolishError(rc, "synthetic data could not be written")
        return fa, [s1, s2]

    def write_truth(self, path):
        lib().pp_synth_write_fasta(self.h, str(path).encode(), 1)

    def fasta(self):
        f = Fasta.__new__(Fasta)
        f.h = lib().pp_synth_fasta(self.h)
        f.view = Contigs()
        lib().pp_fasta_view(f.h, C.byref(f.view))
        n = f.view.n_contigs
        f.names = [lib().pp_fasta_name(f.h, i).decode() for i in range(n)]
        f.descriptions = [lib().pp_fasta_description(f.h, i).decode() for i in range(n)]
        f.off = np.ctypeslib.as_array(C.cast(f.view.off, C.POINTER(C.c_uint64)), shape=(n + 1,)).copy()
        return f

    def pack(self, fasta=None, careful=False):
        """The packed SoA of both mates (mate-1 file then mate-2 file) without materialising SAM text on disk."""
        fasta = fasta or self.fasta()
        p = Packed(fasta, careful)
        for mate in (1, 2):
            rc = lib().pp_synth_feed_pack(self.h, mate, p.h)
            p._check(rc)
        p.finish()
        return p

    def close(self):
        if self.h:
            lib().pp_synth_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- contig sharding across GPUs (csrc/shard.cpp) ---------------------------------------------------------------
class Shards:
    """pp_shards_build: whole contigs per shard, alignments in SAM order, foreign records of a read as ghosts."""

    def __init__(self, contigs, alns, n_shards, shard_of_contig=None, only_shard=-1):
        L = lib()
        L.pp_shards_build.restype = C.c_void_p
        L.pp_shards_build.argtypes = [C.POINTER(Contigs), C.POINTER(Alignments), C.c_uint32]
        L.pp_shards_build_assigned.restype = C.c_void_p
        L.pp_shards_build_assigned.argtypes = [C.POINTER(Contigs), C.POINTER(Alignments), C.c_uint32, C.POINTER(C.c_uint32), C.c_int32]
        L.pp_shards_free.argtypes = [C.c_void_p]
        L.pp_shards_get.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(Contigs), C.POINTER(Alignments),
                                    C.POINTER(C.POINTER(C.c_uint32)), C.POINTER(C.c_uint64)]
        self.n = n_shards
        arr = None
        if shard_of_contig is not None:
            arr = (C.c_uint32 * len(shard_of_contig))(*[int(x) for x in shard_of_contig])
        self.h = L.pp_shards_build_assigned(C.byref(contigs), C.byref(alns), n_shards, arr, only_shard)
        if not self.h:
            raise PolypolishError(PP_ERR_ARG, "pp_shards_build failed")

    def get(self, i):
        """(contigs view, alignments view, original contig indices, number of home alignments)"""
        c, a = Contigs(), Alignments()
        cmap = C.POINTER(C.c_uint32)()
        nh = C.c_uint64()
        rc = lib().pp_shards_get(self.h, i, C.byref(c), C.byref(a), C.byref(cmap), C.byref(nh))
        if rc != PP_OK:
            raise PolypolishError(rc, "pp_shards_get failed")
        return c, a, [cmap[k] for k in range(c.n_contigs)], nh.value

    def close(self):
        if self.h:
            lib().pp_shards_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def view_arrays(v):
    """numpy views of a pp_alignments view (valid while its owner lives)."""
    n = v.n_aln

    def arr(ptr, ct, cnt):
        if cnt == 0 or not ptr:
            return np.zeros(0, dtype=ct)
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), shape=(cnt,))
    return dict(contig=arr(v.contig, C.c_uint32, n), ref_start=arr(v.ref_start, C.c_uint32, n),
                read_id=arr(v.read_id, C.c_uint32, n), seq_off=arr(v.seq_off, C.c_uint32, n),
                seq_len=arr(v.seq_len, C.c_uint16, n), cigar_off=arr(v.cigar_off, C.c_uint32, n),
                n_cigar=arr(v.n_cigar, C.c_uint16, n), nm=arr(v.nm, C.c_uint32, n), flags=arr(v.flags, C.c_uint8, n),
                cigar_ops=arr(v.cigar_ops, C.c_uint32, v.n_cigar_ops), seq_pool=arr(v.seq_pool, C.c_uint8, v.seq_pool_bytes),
                esc_pool=arr(v.esc_pool, C.c_uint8, v.esc_pool_bytes), seq_bits=v.seq_bits, n_reads=v.n_reads)


class TwoBit:
    """pp_alignments_to_2bit: the 2-bit wire format of a 4-bit batch.  `view` shares every array with the source batch (keep it
    alive) except flags, seq_off, seq_pool and esc_pool, which this object owns."""

    def __init__(self, aview):
        L = lib()
        L.pp_alignments_to_2bit.argtypes = [C.POINTER(Alignments), C.POINTER(Alignments), C.POINTER(C.c_void_p)]
        L.pp_2bit_free.argtypes = [C.c_void_p]
        L.pp_2bit_free.restype = None
        self.view = Alignments()
        self.h = C.c_void_p()
        rc = L.pp_alignments_to_2bit(C.byref(aview), C.byref(self.view), C.byref(self.h))
        if rc != PP_OK:
            raise ValueError("pp_alignments_to_2bit: rc %d (the source must be a 4-bit batch)" % rc)
        self._src = aview

    def close(self):
        if self.h:
            lib().pp_2bit_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def polish_files_multi(assembly, sams, devices=None, verbose=False, parser=0, contexts=None, **opts):
    """pp_polish_files_multi: contigs shard over one context per entry of `devices` (entries may repeat), or over the given `contexts`
    (reused across calls like a long-running host would).  parser 0 (default): every context tokenises the text itself and keeps its
    shard (pp_tok_set_shard); 1: host packer + host sharder."""
    L = lib()
    L.pp_polish_files_multi.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_char_p, C.POINTER(C.c_char_p), C.c_int,
                                        C.POINTER(PolishParams), C.c_char_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_int]
    ctxs = contexts if contexts is not None else [Context(d) for d in devices]
    try:
        ctxs[0].set_parser(parser)
        arr_ctx = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
        prm = _params(**opts)
        arr = (C.c_char_p * max(1, len(sams)))(*[str(s).encode() for s in sams])
        out, n = C.c_void_p(), C.c_uint64()
        rc = L.pp_polish_files_multi(arr_ctx, len(ctxs), str(assembly).encode(), arr, len(sams), C.byref(prm), None,
                                     C.byref(out), C.byref(n), int(verbose))
        if rc != PP_OK:
            raise ctxs[0]._err(rc)
        data = C.string_at(out, n.value)
        L.pp_free(out)
        return data
    finally:
        if contexts is None:
            for c in ctxs:
                c.close()
