"""kaiju_b200 -- B200-native Kaiju classification path (host-side Python mirror of include/kaiju_b200.h).

The product is the C-ABI shared library ``kaiju_b200/libkaijub200.so`` (CUDA, sm_100a).  This module only
binds it with ctypes; there is no Python or CPU implementation of the path, and importing the binding on a
machine without the built library raises immediately.

Reference seam mirrored here: ``ConsumerThread`` + ``Config`` (src/ConsumerThread.hpp:64-121,
src/Config.hpp:31-66) -- construct once with the index/taxonomy/parameters, then classify batches of reads.
"""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KJ_B200_LIB") or os.path.join(_HERE, "libkaijub200.so")   # KJ_B200_LIB: A/B builds of the same library

MEM, GREEDY = 0, 1


class KjParams(C.Structure):
    _fields_ = [("mode", C.c_int32), ("min_fragment_length", C.c_uint32), ("mismatches", C.c_uint32),
                ("min_score", C.c_uint32), ("seed_length", C.c_uint32), ("use_evalue", C.c_int32),
                ("min_evalue", C.c_double), ("seg", C.c_int32), ("input_is_protein", C.c_int32), ("name_mode", C.c_int32)]


class KjIndexView(C.Structure):
    _fields_ = [("alen", C.c_int32), ("alphabet", C.c_char_p), ("bwtlen", C.c_int64), ("bwt", C.c_void_p),
                ("startLcode", C.c_void_p), ("db_len", C.c_int64), ("nseq", C.c_int32), ("ncheck", C.c_int64),
                ("chpt_exp", C.c_int32), ("nbytes", C.c_int32), ("pbits", C.c_int32), ("sa", C.c_void_p),
                ("seq_taxon", C.c_void_p), ("seq_accession", C.c_void_p)]


class KjTaxonomyView(C.Structure):
    _fields_ = [("n", C.c_uint64), ("node", C.c_void_p), ("parent", C.c_void_p)]


class KjTableOpts(C.Structure):
    _fields_ = [("rank", C.c_char_p), ("min_percent", C.c_double), ("min_read_count", C.c_int32), ("expand_viruses", C.c_int32),
                ("filter_unclassified", C.c_int32), ("full_path", C.c_int32), ("rank_list", C.c_char_p)]


class KjMkfmiOpts(C.Structure):
    _fields_ = [("chpt_exp", C.c_int32), ("alphabet", C.c_char_p), ("write_bwt_sa", C.c_int32)]


class KjMkfmiStats(C.Structure):
    _fields_ = [("bwtlen", C.c_int64), ("nseq", C.c_int32), ("sort_rounds", C.c_int32), ("round_items", C.c_uint64 * 40),
                ("sort_bytes", C.c_uint64), ("parse_ms", C.c_double), ("upload_ms", C.c_double), ("sort_ms", C.c_double),
                ("assemble_ms", C.c_double), ("write_ms", C.c_double)]


class KaijuError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libkaijub200.so; fails loudly if the CUDA library has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KaijuError("kaiju_b200: %s is missing -- build it with `make -C kaiju_b200/csrc` "
                             "(or python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.kj_last_error.restype = C.c_char_p
        L.kj_fmi_load.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.kj_fmi_view.argtypes = [C.c_void_p, C.POINTER(KjIndexView)]
        L.kj_fmi_free.argtypes = [C.c_void_p]
        L.kj_nodes_load.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.kj_nodes_view.argtypes = [C.c_void_p, C.POINTER(KjTaxonomyView)]
        L.kj_nodes_free.argtypes = [C.c_void_p]
        L.kj_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(KjParams), C.POINTER(KjIndexView), C.POINTER(KjTaxonomyView)]
        if hasattr(L, "kj_create_scaled"):      # (A/B runs may load an older build of the library)
            L.kj_create_scaled.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(KjParams), C.POINTER(KjIndexView), C.POINTER(KjTaxonomyView), C.c_uint32]
            L.kj_index_build_ms.restype = C.c_double; L.kj_index_build_ms.argtypes = [C.c_void_p]
            L.kj_debug_index_checksums.argtypes = [C.c_void_p, C.c_void_p]
            L.kj_debug_host_index_checksums.argtypes = [C.POINTER(KjIndexView), C.POINTER(KjTaxonomyView), C.c_void_p]
            L.kj_classify_multi.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
            L.kj_device_count.restype = C.c_int
            L.kj_classify2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
            L.kj_classify_device2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kj_native_index_write.argtypes = [C.POINTER(KjIndexView), C.POINTER(KjTaxonomyView), C.c_char_p]
        L.kj_create_from_native.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(KjParams), C.c_char_p]
        L.kj_set_params.argtypes = [C.c_void_p, C.POINTER(KjParams)]
        L.kj_destroy.argtypes = [C.c_void_p]
        L.kj_classify.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]
        L.kj_classify_verbose.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kj_classify_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
        L.kj_kernel_launches.restype = C.c_uint64; L.kj_kernel_launches.argtypes = [C.c_void_p]
        L.kj_index_bytes.restype = C.c_uint64; L.kj_index_bytes.argtypes = [C.c_void_p]
        L.kj_last_kernel_ms.restype = C.c_double; L.kj_last_kernel_ms.argtypes = [C.c_void_p]
        L.kj_classify_files.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.kj_counts_reset.argtypes = [C.c_void_p]
        L.kj_counts_size.restype = C.c_uint64; L.kj_counts_size.argtypes = [C.c_void_p]
        L.kj_counts_device_ptr.restype = C.c_void_p; L.kj_counts_device_ptr.argtypes = [C.c_void_p]
        L.kj_counts_add_device.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]
        L.kj_counts_get.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.kj_table_write.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(KjTableOpts), C.c_char_p, C.c_int]
        L.kj_counts_table.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(KjTableOpts), C.c_char_p, C.c_int]
        L.kj_check_errors.argtypes = [C.c_void_p]
        L.kj_launch_geometry.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.kj_version.restype = C.c_int
        if hasattr(L, "kj_mkfmi"):
            L.kj_mkfmi.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(KjMkfmiOpts), C.c_int, C.POINTER(KjMkfmiStats)]
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise KaijuError("kaiju_b200 error %d: %s" % (rc, lib().kj_last_error().decode()))


def make_params(mode="mem", m=11, e=3, s=65, seed=7, E=0.01, seg=True, use_evalue=None, protein=False, name_mode=False):
    """Config fields as the kaiju CLI sets them (kaiju.cpp:74-202): -a -m -e -s -l -E -x/-X -p."""
    greedy = mode in ("greedy", GREEDY, 1)
    if use_evalue is None:
        use_evalue = greedy
    return KjParams(mode=1 if greedy else 0, min_fragment_length=m, mismatches=e, min_score=s, seed_length=seed,
                    use_evalue=1 if (use_evalue and greedy) else 0, min_evalue=E, seg=1 if seg else 0, input_is_protein=1 if protein else 0, name_mode=1 if name_mode else 0)


def _table_opts(rank, min_percent=0.0, min_read_count=0, expand_viruses=False, filter_unclassified=False, full_path=False, rank_list=None):
    return KjTableOpts(rank.encode(), float(min_percent), int(min_read_count), int(expand_viruses), int(filter_unclassified), int(full_path),
                       rank_list.encode() if rank_list else None)


def write_table(taxon_ids, counts, nodes_path, names_path, label, out_path, rank="species", append=False, **kw):
    """kaiju2table's report from per-taxon read counts (taxon id 0 = unclassified reads).  Host-only, no GPU needed."""
    ids = np.ascontiguousarray(taxon_ids, dtype=np.uint64); cnt = np.ascontiguousarray(counts, dtype=np.uint64)
    o = _table_opts(rank, **kw)
    _check(lib().kj_table_write(ids.ctypes.data, cnt.ctypes.data, len(ids), nodes_path.encode(), names_path.encode(), label.encode(), C.byref(o),
                                out_path.encode(), 1 if append else 0))


def host_index_checksums(fmi_path, nodes_path):
    """Test hook: the checksums Classifier.debug_index_checksums() must report, from the host transcoder (no GPU needed)."""
    L = lib(); fmi = C.c_void_p(); nodes = C.c_void_p(); out = np.zeros(8, dtype=np.uint64)
    _check(L.kj_fmi_load(fmi_path.encode(), C.byref(fmi)))
    try:
        _check(L.kj_nodes_load(nodes_path.encode(), C.byref(nodes)))
        try:
            iv = KjIndexView(); tv = KjTaxonomyView(); L.kj_fmi_view(fmi, C.byref(iv)); L.kj_nodes_view(nodes, C.byref(tv))
            _check(L.kj_debug_host_index_checksums(C.byref(iv), C.byref(tv), out.ctypes.data))
        finally:
            L.kj_nodes_free(nodes)
    finally:
        L.kj_fmi_free(fmi)
    return out


def write_native_index(fmi_path, nodes_path, out_path):
    """Transcode a reference .fmi + nodes.dmp once into the device-native index file (no GPU needed)."""
    L = lib(); fmi = C.c_void_p(); nodes = C.c_void_p()
    _check(L.kj_fmi_load(fmi_path.encode(), C.byref(fmi)))
    try:
        _check(L.kj_nodes_load(nodes_path.encode(), C.byref(nodes)))
        try:
            iv = KjIndexView(); tv = KjTaxonomyView(); L.kj_fmi_view(fmi, C.byref(iv)); L.kj_nodes_view(nodes, C.byref(tv))
            _check(L.kj_native_index_write(C.byref(iv), C.byref(tv), out_path.encode()))
        finally:
            L.kj_nodes_free(nodes)
    finally:
        L.kj_fmi_free(fmi)


def build_index(faa, prefix, exponent=3, alphabet="ACDEFGHIKLMNPQRSTVWY", device=0, write_bwt_sa=False):
    """Protein FASTA -> <prefix>.fmi on the GPU, byte for byte what `kaiju-mkbwt -a ALPHABET -e EXPONENT` + `kaiju-mkfmi` write
    (kj_mkfmi; alphabet may also be "protein").  With write_bwt_sa also <prefix>.bwt and <prefix>.sa.  Returns the build statistics."""
    o = KjMkfmiOpts(int(exponent), alphabet.encode() if alphabet else None, 1 if write_bwt_sa else 0); st = KjMkfmiStats()
    _check(lib().kj_mkfmi(os.fspath(faa).encode(), os.fspath(prefix).encode(), C.byref(o), int(device), C.byref(st)))
    return {"bwtlen": int(st.bwtlen), "nseq": int(st.nseq), "sort_rounds": int(st.sort_rounds),
            "round_items": [int(st.round_items[i]) for i in range(st.sort_rounds)], "sort_bytes": int(st.sort_bytes),
            "parse_ms": st.parse_ms, "upload_ms": st.upload_ms, "sort_ms": st.sort_ms, "assemble_ms": st.assemble_ms, "write_ms": st.write_ms}


def device_count():
    return int(lib().kj_device_count())


def classify_multi(classifiers, seq1, off1, seq2=None, off2=None, want_best=True):
    """One batch over several Classifiers (one per GPU, same index and parameters) in this process: contiguous shards, results in
    input order (kj_classify_multi -- the counterpart of the reference's `-z N`)."""
    n = len(off1) - 1
    seq1 = np.ascontiguousarray(seq1, dtype=np.uint8); off1 = np.ascontiguousarray(off1, dtype=np.uint64)
    p2 = o2 = None
    if seq2 is not None:
        seq2 = np.ascontiguousarray(seq2, dtype=np.uint8); off2 = np.ascontiguousarray(off2, dtype=np.uint64)
        p2, o2 = seq2.ctypes.data, off2.ctypes.data
    tax = np.zeros(n, dtype=np.uint64); best = np.zeros(n, dtype=np.uint32) if want_best else None
    arr = (C.c_void_p * len(classifiers))(*[c._ctx for c in classifiers])
    _check(lib().kj_classify_multi(arr, len(classifiers), seq1.ctypes.data, off1.ctypes.data, p2, o2, n, tax.ctypes.data, best.ctypes.data if want_best else None))
    return (tax, best) if want_best else tax


class Classifier:
    """One GPU context: the .fmi index and nodes.dmp taxonomy resident in HBM + run parameters.
    `Classifier(native_path, None)` loads a device-native index file written by write_native_index()."""

    def __init__(self, fmi_path, nodes_path, device=0, params=None, copies=1, **kw):
        """copies > 1: the index of the collection in which every sequence occurs `copies` times (kj_create_scaled)."""
        L = lib()
        self._ctx = C.c_void_p()
        if nodes_path is None:
            self.params = params if params is not None else make_params(**kw)
            _check(L.kj_create_from_native(C.byref(self._ctx), device, C.byref(self.params), fmi_path.encode()))
            self.device = device; self.bwtlen = self.nseq = None
            return
        fmi = C.c_void_p(); nodes = C.c_void_p()
        _check(L.kj_fmi_load(fmi_path.encode(), C.byref(fmi)))
        try:
            _check(L.kj_nodes_load(nodes_path.encode(), C.byref(nodes)))
            try:
                iv = KjIndexView(); tv = KjTaxonomyView()
                L.kj_fmi_view(fmi, C.byref(iv)); L.kj_nodes_view(nodes, C.byref(tv))
                self.params = params if params is not None else make_params(**kw)
                self.bwtlen = int(iv.bwtlen); self.nseq = int(iv.nseq)
                self.bwtlen *= int(copies); self.nseq *= int(copies)
                if int(copies) == 1:
                    _check(L.kj_create(C.byref(self._ctx), device, C.byref(self.params), C.byref(iv), C.byref(tv)))
                else:
                    _check(L.kj_create_scaled(C.byref(self._ctx), device, C.byref(self.params), C.byref(iv), C.byref(tv), int(copies)))
            finally:
                L.kj_nodes_free(nodes)
        finally:
            L.kj_fmi_free(fmi)
        self.device = device

    def set_params(self, params=None, **kw):
        self.params = params if params is not None else make_params(**kw)
        _check(lib().kj_set_params(self._ctx, C.byref(self.params)))

    def close(self):
        if self._ctx:
            lib().kj_destroy(self._ctx); self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- host buffers (numpy): H2D + kernel + D2H inside, like handing ReadItems to the consumer threads
    def classify(self, seq1, off1, seq2=None, off2=None, want_best=True):
        n = len(off1) - 1
        seq1 = np.ascontiguousarray(seq1, dtype=np.uint8); off1 = np.ascontiguousarray(off1, dtype=np.uint64)
        p2 = o2 = None
        if seq2 is not None:
            seq2 = np.ascontiguousarray(seq2, dtype=np.uint8); off2 = np.ascontiguousarray(off2, dtype=np.uint64)
            p2, o2 = seq2.ctypes.data, off2.ctypes.data
        tax = np.zeros(n, dtype=np.uint64); best = np.zeros(n, dtype=np.uint32) if want_best else None
        _check(lib().kj_classify(self._ctx, seq1.ctypes.data, off1.ctypes.data, p2, o2, n, tax.ctypes.data,
                                 best.ctypes.data if want_best else None))
        return (tax, best) if want_best else tax

    def classify_verbose(self, seq1, off1, seq2=None, off2=None):
        """taxon, best, and the ascending match-id set per read (columns 3-5 of `kaiju -v`)."""
        n = len(off1) - 1
        seq1 = np.ascontiguousarray(seq1, dtype=np.uint8); off1 = np.ascontiguousarray(off1, dtype=np.uint64)
        p2 = o2 = None
        if seq2 is not None:
            seq2 = np.ascontiguousarray(seq2, dtype=np.uint8); off2 = np.ascontiguousarray(off2, dtype=np.uint64)
            p2, o2 = seq2.ctypes.data, off2.ctypes.data
        tax = np.zeros(n, dtype=np.uint64); best = np.zeros(n, dtype=np.uint32)
        ids = np.zeros((n, 21), dtype=np.uint64); nids = np.zeros(n, dtype=np.uint8)
        _check(lib().kj_classify_verbose(self._ctx, seq1.ctypes.data, off1.ctypes.data, p2, o2, n, tax.ctypes.data, best.ctypes.data,
                                         ids.ctypes.data, nids.ctypes.data))
        return tax, best, [tuple(int(x) for x in ids[i, :nids[i]]) for i in range(n)]

    def classify_ptrs(self, seq1_ptr, off1_ptr, seq2_ptr, off2_ptr, n, tax_ptr, best_ptr):
        """Host pointers (e.g. pinned torch tensors' data_ptr())."""
        _check(lib().kj_classify(self._ctx, seq1_ptr, off1_ptr, seq2_ptr, off2_ptr, n, tax_ptr, best_ptr))

    # ---- device buffers (raw device pointers, e.g. torch tensors' data_ptr()); asynchronous on `stream`
    def classify_device(self, d_seq1, d_off1, d_seq2, d_off2, n, d_tax, d_best=None, max_len1=0, max_len2=0, stream=None):
        _check(lib().kj_classify_device(self._ctx, d_seq1, d_off1, d_seq2, d_off2, n, max_len1, max_len2, d_tax, d_best, stream))

    def classify_device2(self, d_seq1, d_off1, d_seq2, d_off2, n, d_tax, d_best, d_compact, max_len1=0, max_len2=0, stream=None):
        """As classify_device, plus a device uint32 array of dense taxon indices (see compact_ids); d_tax may be None."""
        _check(lib().kj_classify_device2(self._ctx, d_seq1, d_off1, d_seq2, d_off2, n, max_len1, max_len2, d_tax, d_best, d_compact, stream))

    def classify2_ptrs(self, seq1_ptr, off1_ptr, seq2_ptr, off2_ptr, n, tax_ptr, best_ptr, d_compact):
        """Host buffers in and out (kj_classify) plus the dense taxon indices left in the DEVICE array d_compact."""
        _check(lib().kj_classify2(self._ctx, seq1_ptr, off1_ptr, seq2_ptr, off2_ptr, n, tax_ptr, best_ptr, d_compact))

    def compact_ids(self):
        """NCBI taxon id of every dense taxon index (the id list of counts(); the last entry, 0, stands for unclassified)."""
        return self.counts(nonzero=False)[0]

    def classify_files(self, in1, in2=None, out_path=None, verbose=False):
        """FASTA/FASTQ(.gz) files -> kaiju output file, parsed / classified / formatted on the device.  Returns (reads, classified)."""
        n = C.c_uint64(); k = C.c_uint64()
        _check(lib().kj_classify_files(self._ctx, in1.encode(), in2.encode() if in2 else None, out_path.encode() if out_path else None,
                                       1 if verbose else 0, C.byref(n), C.byref(k)))
        return int(n.value), int(k.value)

    # ---- per-taxon read counts accumulated in HBM by the successful classify calls (input of kaiju2table)
    def counts_reset(self):
        _check(lib().kj_counts_reset(self._ctx))

    def counts(self, nonzero=True):
        """(taxon ids, read counts); the last entry (id 0) counts the unclassified reads."""
        n = int(lib().kj_counts_size(self._ctx)); ids = np.zeros(n, dtype=np.uint64); cnt = np.zeros(n, dtype=np.uint64)
        _check(lib().kj_counts_get(self._ctx, ids.ctypes.data, cnt.ctypes.data))
        if nonzero:
            k = cnt != 0; return ids[k], cnt[k]
        return ids, cnt

    def counts_add_device(self, d_tax, n, stream=None):
        _check(lib().kj_counts_add_device(self._ctx, d_tax, n, stream))

    @property
    def counts_device_ptr(self):
        return lib().kj_counts_device_ptr(self._ctx), int(lib().kj_counts_size(self._ctx))

    def counts_table(self, nodes_path, names_path, label, out_path, rank="species", append=False, **kw):
        """kaiju2table's report for the reads counted so far."""
        o = _table_opts(rank, **kw)
        _check(lib().kj_counts_table(self._ctx, nodes_path.encode(), names_path.encode(), label.encode(), C.byref(o), out_path.encode(), 1 if append else 0))

    def check_errors(self):
        _check(lib().kj_check_errors(self._ctx))

    @property
    def kernel_launches(self):
        return int(lib().kj_kernel_launches(self._ctx))

    @property
    def index_bytes(self):
        return int(lib().kj_index_bytes(self._ctx))

    @property
    def index_build_ms(self):
        return float(lib().kj_index_build_ms(self._ctx))

    def debug_index_checksums(self):
        out = np.zeros(8, dtype=np.uint64); _check(lib().kj_debug_index_checksums(self._ctx, out.ctypes.data)); return out

    @property
    def last_kernel_ms(self):
        return float(lib().kj_last_kernel_ms(self._ctx))

    @property
    def launch_geometry(self):
        g = C.c_int(); b = C.c_int(); s = C.c_int()
        lib().kj_launch_geometry(self._ctx, C.byref(g), C.byref(b), C.byref(s))
        return g.value, b.value, s.value
