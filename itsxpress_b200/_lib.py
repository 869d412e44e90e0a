"""ctypes binding of libitsx_b200.so (C ABI: include/itsx_b200.h).

The library is the product: if it is missing or no B200 is present the calls below raise -- there
is no CPU fallback anywhere in this package.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# ITSX_B200_LIB: an experimental build of the same library (tools/build_variant.py); never another implementation
LIB_PATH = os.environ.get("ITSX_B200_LIB") or os.path.join(_HERE, "libitsx_b200.so")
_LIB = None

MAXM = 45
MAXDOM = 8


class ItsxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libitsx_b200 error %d: %s" % (code, msg))
        self.code = code


class SearchParams(C.Structure):
    _fields_ = [("T", C.c_float), ("F1", C.c_double), ("F2", C.c_double), ("F3", C.c_double), ("domE", C.c_double),
                ("resolve_multidomain", C.c_int32), ("keep_rows", C.c_int32), ("domz_upper", C.c_int64)]


class SearchStats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("n_seq", "n_prof", "n_pairs", "n_past_msv", "n_past_bias", "n_past_fwd",
                                          "n_hits_reported", "n_domains", "n_domains_reported",
                                          "n_multidomain_regions", "n_dom_overflow")] + \
               [(n, C.c_double) for n in ("msv_cells", "bias_rows", "fwd_cells", "bck_cells", "env_cells")] + \
               [(n, C.c_float) for n in ("ms_msv", "ms_bias", "ms_fwd", "ms_mdom", "ms_env", "ms_final", "ms_total",
                                          "reserved")] + \
               [("n_selected_multidomain", C.c_int64), ("n_vit_run", C.c_int64), ("n_past_vit", C.c_int64),
                ("vit_cells", C.c_double), ("ms_vit", C.c_float), ("reserved2", C.c_float)]

    def asdict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class DerepStats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("n_reads", "n_unique", "n_collided", "bytes_ascii")] + \
               [(n, C.c_float) for n in ("ms_pack", "ms_hash", "ms_insert", "ms_verify", "ms_compact", "ms_total")]

    def asdict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class ClusterParams(C.Structure):
    _fields_ = [("id", C.c_double), ("strand_both", C.c_int32), ("per_sample", C.c_int32)]


class ClusterStats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("n_unique", "n_centroids", "n_segments", "n_candidates", "n_verified",
                                          "n_accepted", "n_rounds")] + \
               [("d_max", C.c_int32), ("n_len_slots", C.c_int32)] + \
               [(n, C.c_float) for n in ("ms_index", "ms_candidates", "ms_verify", "ms_resolve", "ms_remap", "ms_total")]

    def asdict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class MergeParams(C.Structure):
    _fields_ = [("maxdiffs", C.c_int32), ("allow_stagger", C.c_int32), ("qmax", C.c_int32), ("minovlen", C.c_int32),
                ("qmaxout", C.c_int32), ("qminout", C.c_int32), ("ascii", C.c_int32), ("reserved", C.c_int32),
                ("maxee", C.c_double), ("maxdiffpct", C.c_double)]


class MergeStats(C.Structure):
    _fields_ = [("n_pairs", C.c_int64), ("n_merged", C.c_int64), ("by_reason", C.c_int64 * 16),
                ("bytes_in", C.c_int64), ("bytes_out", C.c_int64), ("ms_kernel", C.c_float)]


MERGE_REASONS = ("ok", "repeat", "staggered", "maxdiffs", "maxdiffpct", "nokmers", "minscore", "minovlen", "maxee",
                 "badqual")


class RunStats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("n_reads", "n_unique", "n_kept", "out_bytes")] + \
               [(n, C.c_float) for n in ("ms_h2d", "ms_derep", "ms_search", "ms_trim", "ms_d2h", "ms_total",
                                          "ms_gather", "reserved")]

    def asdict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


ROW_DTYPE = np.dtype([
    ("seq", "<i4"), ("prof", "<i4"), ("ienv", "<i4"), ("jenv", "<i4"), ("tlen", "<i4"), ("dom_idx", "<i4"),
    ("bitscore", "<f4"), ("envsc", "<f4"), ("domcorrection", "<f4"), ("seq_score", "<f4"),
    ("lnP", "<f8"), ("seq_lnP", "<f8"), ("is_multidomain", "<i4"), ("reported", "<i4"),
])

# every symbol include/itsx_b200.h declares (tests check that the .so exports all of them)
SYMBOLS = [
    "itsx_create", "itsx_destroy", "itsx_last_error", "itsx_device_info", "itsx_stream", "itsx_sync",
    "itsx_pinned_alloc", "itsx_pinned_free",
    "itsx_profiles_clear", "itsx_profiles_append_file", "itsx_profiles_count", "itsx_profile_name", "itsx_profile_M",
    "itsx_profiles_set_sides", "itsx_profile_msv",
    "itsx_derep", "itsx_derep_clusters", "itsx_derep_unique_keys", "itsx_derep_get_stats", "itsx_derep_set_key_bits",
    "itsx_search_default_params", "itsx_search", "itsx_search_seqs", "itsx_search_get_stats", "itsx_hits",
    "itsx_nreported", "itsx_positions", "itsx_search_stage1", "itsx_search_seqs_stage1", "itsx_search_shard",
    "itsx_nreported_set", "itsx_search_stage2", "itsx_positions_set",
    "itsx_trim_set_map", "itsx_trim_bounds", "itsx_trim_gather", "itsx_run", "itsx_reads_upload", "itsx_run_resident",
    "itsx_launch_count", "itsx_reads_begin", "itsx_reads_append", "itsx_reads_end", "itsx_trim_gather_range",
    "itsx_derep_map", "itsx_reads_set_samples", "itsx_trim_gather_resident", "itsx_run_trim", "itsx_quals_upload", "itsx_derep_resident", "itsx_run_fetch",
    "itsx_shard_plan", "itsx_shard_pack", "itsx_shard_owner_derep", "itsx_shard_answers", "itsx_shard_apply",
    "itsx_merge_default_params", "itsx_merge_pairs", "itsx_merge_fetch", "itsx_merge_get_stats",
    "itsx_gzip_bound", "itsx_gzip_compress",
    "itsx_gz_open", "itsx_gz_read", "itsx_gz_eof", "itsx_gz_close", "itsx_gz_tune", "itsx_gz_stat",
    "itsx_host_last_error", "itsx_fastq_index", "itsx_fastq_cut", "itsx_bytes_gather", "itsx_fastq_format", "itsx_domtbl_format",
    "itsx_fastq_labels", "itsx_uc_format", "itsx_repfa_format",
    "itsx_cluster", "itsx_cluster_fetch", "itsx_cluster_get_stats", "itsx_cluster_dtable", "itsx_cluster_set_key_bits",
]


def lib():
    """Load the shared library (built in-tree by itsxpress_b200.build)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise ImportError("libitsx_b200.so is not built: run `python -m itsxpress_b200.build` "
                          "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.itsx_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.itsx_destroy.argtypes = [vp]
    L.itsx_destroy.restype = None
    L.itsx_last_error.argtypes = [vp]
    L.itsx_last_error.restype = C.c_char_p
    L.itsx_device_info.argtypes = [vp, vp, vp, vp, vp]
    L.itsx_stream.argtypes = [vp]
    L.itsx_stream.restype = vp
    L.itsx_sync.argtypes = [vp]
    L.itsx_pinned_alloc.argtypes = [C.c_size_t]
    L.itsx_pinned_alloc.restype = vp
    L.itsx_pinned_free.argtypes = [vp]
    L.itsx_pinned_free.restype = None
    L.itsx_profiles_clear.argtypes = [vp]
    L.itsx_profiles_append_file.argtypes = [vp, C.c_char_p, C.POINTER(C.c_char_p), C.c_int]
    L.itsx_profiles_count.argtypes = [vp]
    L.itsx_profile_name.argtypes = [vp, C.c_int]
    L.itsx_profile_name.restype = C.c_char_p
    L.itsx_profile_M.argtypes = [vp, C.c_int]
    L.itsx_profiles_set_sides.argtypes = [vp, vp, C.c_int]
    L.itsx_profile_msv.argtypes = [vp, C.c_int, vp, vp]
    L.itsx_derep.argtypes = [vp, vp, vp, i64, vp, vp, vp]
    L.itsx_derep_clusters.argtypes = [vp, vp, vp]
    L.itsx_derep_unique_keys.argtypes = [vp, vp]
    L.itsx_derep_get_stats.argtypes = [vp, C.POINTER(DerepStats)]
    L.itsx_derep_set_key_bits.argtypes = [vp, C.c_int]
    L.itsx_cluster.argtypes = [vp, C.POINTER(ClusterParams), vp, vp]
    L.itsx_cluster_fetch.argtypes = [vp, vp, vp, vp, vp]
    L.itsx_cluster_get_stats.argtypes = [vp, C.POINTER(ClusterStats)]
    L.itsx_cluster_dtable.argtypes = [C.c_double, i32, vp]
    L.itsx_cluster_set_key_bits.argtypes = [vp, C.c_int]
    L.itsx_search_default_params.argtypes = [C.POINTER(SearchParams)]
    L.itsx_search_default_params.restype = None
    L.itsx_search.argtypes = [vp, C.POINTER(SearchParams)]
    L.itsx_search_seqs.argtypes = [vp, vp, vp, i64, C.POINTER(SearchParams)]
    L.itsx_search_get_stats.argtypes = [vp, C.POINTER(SearchStats)]
    L.itsx_hits.argtypes = [vp, vp, i64, vp]
    L.itsx_nreported.argtypes = [vp, vp]
    L.itsx_positions.argtypes = [vp] + [vp] * 9
    L.itsx_search_stage1.argtypes = [vp, C.POINTER(SearchParams)]
    L.itsx_search_seqs_stage1.argtypes = [vp, vp, vp, i64, C.POINTER(SearchParams)]
    L.itsx_search_shard.argtypes = [vp, i64, i64]
    L.itsx_nreported_set.argtypes = [vp, vp]
    L.itsx_search_stage2.argtypes = [vp]
    L.itsx_positions_set.argtypes = [vp, vp, vp, vp, i64]
    L.itsx_trim_set_map.argtypes = [vp, vp, i64, i64]
    L.itsx_trim_bounds.argtypes = [vp, C.c_int, vp, i64, vp, vp, vp, vp]
    L.itsx_trim_gather.argtypes = [vp, C.c_int, vp, vp, vp, i64, vp, vp]
    L.itsx_run.argtypes = [vp, vp, vp, i64, C.POINTER(SearchParams), vp, vp, vp, vp, C.POINTER(RunStats)]
    L.itsx_reads_upload.argtypes = [vp, vp, vp, i64]
    L.itsx_run_resident.argtypes = [vp, C.POINTER(SearchParams), C.POINTER(RunStats)]
    L.itsx_launch_count.argtypes = [vp]
    L.itsx_launch_count.restype = i64
    L.itsx_reads_set_samples.argtypes = [vp, vp, i32]
    L.itsx_derep_map.argtypes = [vp, vp, vp, vp]
    L.itsx_reads_begin.argtypes = [vp, i64, i64]
    L.itsx_reads_append.argtypes = [vp, vp, vp, vp, i64]
    L.itsx_reads_end.argtypes = [vp, vp, vp]
    L.itsx_trim_gather_range.argtypes = [vp, C.c_int, i64, i64, vp, vp]
    L.itsx_trim_gather_resident.argtypes = [vp, C.c_int, vp, vp]
    L.itsx_run_trim.argtypes = [vp, vp, vp, vp, i64, C.POINTER(SearchParams), vp, vp, vp, vp, vp, C.POINTER(RunStats)]
    L.itsx_quals_upload.argtypes = [vp, vp]
    L.itsx_derep_resident.argtypes = [vp, C.c_int, vp]
    L.itsx_run_fetch.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.itsx_shard_plan.argtypes = [vp, C.c_int, vp, vp]
    L.itsx_shard_pack.argtypes = [vp, i64, vp, vp]
    L.itsx_shard_owner_derep.argtypes = [vp, vp, i64, vp, i64, vp]
    L.itsx_shard_answers.argtypes = [vp, i64, vp]
    L.itsx_shard_apply.argtypes = [vp, vp, i64, vp, vp]
    L.itsx_merge_default_params.argtypes = [C.POINTER(MergeParams)]
    L.itsx_merge_default_params.restype = None
    L.itsx_merge_pairs.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, C.POINTER(MergeParams), vp, vp, vp, vp]
    L.itsx_merge_fetch.argtypes = [vp, vp, vp, vp, vp]
    L.itsx_merge_get_stats.argtypes = [vp, C.POINTER(MergeStats)]
    L.itsx_gzip_bound.argtypes = [i64]
    L.itsx_gzip_bound.restype = i64
    L.itsx_gzip_compress.argtypes = [vp, vp, i64, vp, i64, C.POINTER(i64)]
    L.itsx_gz_open.argtypes = [vp, i64, C.c_int]
    L.itsx_gz_open.restype = vp
    L.itsx_gz_read.argtypes = [vp, vp, i64, i64]
    L.itsx_gz_read.restype = i64
    L.itsx_gz_eof.argtypes = [vp]
    L.itsx_gz_close.argtypes = [vp]
    L.itsx_gz_close.restype = None
    L.itsx_gz_tune.argtypes = [vp, i64, i64, i64]
    L.itsx_gz_stat.argtypes = [vp, C.c_int]
    L.itsx_gz_stat.restype = i64
    L.itsx_host_last_error.restype = C.c_char_p
    L.itsx_domtbl_format.restype = i64
    L.itsx_domtbl_format.argtypes = [vp, i64, vp, vp, vp, vp, vp, vp, C.c_double, vp, i64]
    L.itsx_fastq_labels.restype = i64
    L.itsx_fastq_labels.argtypes = [vp, vp, vp, i64, vp, vp]
    L.itsx_uc_format.restype = i64
    L.itsx_uc_format.argtypes = [vp, vp, vp, i64, vp, i64, vp, vp, vp, vp, i64]
    L.itsx_repfa_format.restype = i64
    L.itsx_repfa_format.argtypes = [vp, vp, vp, vp, vp, vp, i64, i32, vp, i64]
    L.itsx_fastq_cut.restype = i64
    L.itsx_fastq_cut.argtypes = [vp, i64]
    L.itsx_fastq_index.restype = i64
    L.itsx_fastq_index.argtypes = [vp, i64, i64, vp, vp, vp, vp, vp]
    L.itsx_bytes_gather.restype = i64
    L.itsx_bytes_gather.argtypes = [vp, vp, vp, i64, vp, vp]
    L.itsx_fastq_format.restype = i64
    L.itsx_fastq_format.argtypes = [vp, vp, vp, vp, i64, vp, vp, vp, C.c_char_p, C.c_char_p, i32, C.c_char_p,
                                    C.c_char_p, i32, vp]
    _LIB = L
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def merge_params(allow_stagger=False, **kw):
    """vsearch --fastq_mergepairs options as the reference passes them (SeqSample.py:314-349)."""
    prm = MergeParams()
    lib().itsx_merge_default_params(C.byref(prm))
    prm.allow_stagger = int(bool(allow_stagger))
    for k, v in kw.items():
        setattr(prm, k, v)
    return prm


def cluster_dtable(cluster_id, lmax):
    """D[L] for L = 0 .. lmax: the largest edit distance a pair whose longer member has length L may have and still be
    accepted at identity ``cluster_id`` (the table itsx_cluster uses)."""
    D = np.empty(int(lmax) + 1, np.int32)
    rc = lib().itsx_cluster_dtable(float(cluster_id), int(lmax), _p(D))
    if rc < 0:
        raise ItsxError(rc, "cluster_dtable: id must be in (0.5, 1] and lmax >= 0")
    return D


def default_params():
    prm = SearchParams()
    lib().itsx_search_default_params(C.byref(prm))
    return prm


class PinnedBuffer:
    """Page-locked host memory (cudaHostAlloc) viewed as numpy arrays; freed on close()/collection."""

    def __init__(self, nbytes):
        self.nbytes = max(1, int(nbytes))
        self.ptr = lib().itsx_pinned_alloc(self.nbytes)
        if not self.ptr:
            raise MemoryError("cudaHostAlloc failed")
        self._buf = (C.c_char * self.nbytes).from_address(self.ptr)

    def array(self, dtype=np.uint8, count=None, offset=0):
        dtype = np.dtype(dtype)
        if count is None:
            count = (self.nbytes - offset) // dtype.itemsize
        return np.frombuffer(self._buf, dtype=dtype, count=int(count), offset=int(offset))

    def close(self):
        if self.ptr:
            lib().itsx_pinned_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One GPU context (one per process / per device)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        rc = lib().itsx_create(int(device), C.byref(self._h))
        if rc != 0:
            raise ItsxError(rc, lib().itsx_last_error(None).decode())
        self.device = device
        self.names = []

    def close(self):
        if self._h:
            lib().itsx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc < 0:
            raise ItsxError(rc, lib().itsx_last_error(self._h).decode())
        return rc

    def device_info(self):
        sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
        mem = C.c_int64()
        self._chk(lib().itsx_device_info(self._h, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(mem)))
        return dict(sm_count=sm.value, cc=(ma.value, mi.value), mem_bytes=mem.value)

    @property
    def stream(self):
        return lib().itsx_stream(self._h)

    def sync(self):
        self._chk(lib().itsx_sync(self._h))

    def launch_count(self):
        return int(lib().itsx_launch_count(self._h))

    # ---- profiles --------------------------------------------------------------------------
    def load_profiles(self, paths, prefixes=None, skip_missing=True):
        """Profiles of the given HMMER3 files whose NAME starts with a prefix, in file order."""
        L = lib()
        self._chk(L.itsx_profiles_clear(self._h))
        pre = [p.encode() for p in (prefixes or [])]
        arr = (C.c_char_p * max(1, len(pre)))(*pre) if pre else None
        if isinstance(paths, (str, bytes)):
            paths = [paths]
        for p in paths:
            if skip_missing and not os.path.exists(p):
                continue
            self._chk(L.itsx_profiles_append_file(self._h, os.fsencode(p), arr, len(pre)))
        n = L.itsx_profiles_count(self._h)
        self.names = [L.itsx_profile_name(self._h, i).decode() for i in range(n)]
        return n

    def profile_M(self, p):
        return lib().itsx_profile_M(self._h, p)

    def set_sides(self, side):
        side = np.ascontiguousarray(side, dtype=np.int8)
        self._chk(lib().itsx_profiles_set_sides(self._h, _p(side), len(side)))

    def set_sides_by_prefix(self, left_prefix, right_prefix):
        side = np.full(len(self.names), -1, np.int8)
        for i, nm in enumerate(self.names):
            if nm.startswith(left_prefix):
                side[i] = 0
            elif nm.startswith(right_prefix):
                side[i] = 1
        self.set_sides(side)
        return side

    def profile_msv(self, p):
        M = self.profile_M(p)
        cost = np.zeros((M + 1, 16), np.uint8)
        sc = np.zeros(4, np.int32)
        self._chk(lib().itsx_profile_msv(self._h, p, _p(cost), _p(sc)))
        return cost, dict(bias=int(sc[0]), base=int(sc[1]), tbm=int(sc[2]), tec=int(sc[3]))

    # ---- derep ------------------------------------------------------------------------------
    def derep(self, seq, off):
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.int64)
        n = len(off) - 1
        rep = np.empty(n, np.int32)
        strand = np.empty(n, np.uint8)
        nu = C.c_int64()
        self._chk(lib().itsx_derep(self._h, _p(seq), _p(off), n, _p(rep), _p(strand), C.byref(nu)))
        return rep, strand, int(nu.value)

    def derep_clusters(self, n_unique):
        first = np.empty(n_unique, np.int32)
        ab = np.empty(n_unique, np.int32)
        self._chk(lib().itsx_derep_clusters(self._h, _p(first), _p(ab)))
        return first, ab

    def derep_unique_keys(self, n_unique):
        keys = np.empty(n_unique, np.uint64)
        self._chk(lib().itsx_derep_unique_keys(self._h, _p(keys)))
        return keys

    def derep_map(self, n):
        """(rep_index, strand, uid) of the n resident reads after a derep."""
        rep, strand, uid = np.empty(n, np.int32), np.empty(n, np.uint8), np.empty(n, np.int32)
        self._chk(lib().itsx_derep_map(self._h, _p(rep), _p(strand), _p(uid)))
        return rep, strand, uid

    def derep_stats(self):
        st = DerepStats()
        self._chk(lib().itsx_derep_get_stats(self._h, C.byref(st)))
        return st

    def set_key_bits(self, bits):
        self._chk(lib().itsx_derep_set_key_bits(self._h, int(bits)))

    # ---- clustering ---------------------------------------------------------------------------
    def cluster(self, cluster_id, order=None, per_sample=False):
        """Greedy clustering of the resident derep's classes at identity ``cluster_id`` (itsx_cluster).  ``order``: unique
        indices in processing order (None: abundance descending, then first occurrence).  Returns the centroid count;
        the search set becomes the centroids and the read -> row map their rows.  ``per_sample``: with sample ids set
        (set_samples), cluster every sample on its own; without it sample ids are refused."""
        prm = ClusterParams(float(cluster_id), 1, int(bool(per_sample)))
        o = None if order is None else np.ascontiguousarray(order, dtype=np.int32)
        nc = C.c_int64()
        self._chk(lib().itsx_cluster(self._h, C.byref(prm), _p(o), C.byref(nc)))
        return int(nc.value)

    def cluster_fetch(self, n_unique, n_centroids):
        """(centroid_row_of_unique, strand_of_unique, ed_of_unique, unique_of_row) of the last itsx_cluster."""
        row, strand = np.empty(n_unique, np.int32), np.empty(n_unique, np.uint8)
        ed, uor = np.empty(n_unique, np.int32), np.empty(n_centroids, np.int32)
        self._chk(lib().itsx_cluster_fetch(self._h, _p(row), _p(strand), _p(ed), _p(uor)))
        return row, strand, ed, uor

    def cluster_set_key_bits(self, bits):
        """test hook: itsx_cluster keeps only the low ``bits`` bits of its segment keys (64 = normal)"""
        self._chk(lib().itsx_cluster_set_key_bits(self._h, int(bits)))

    def cluster_stats(self):
        st = ClusterStats()
        self._chk(lib().itsx_cluster_get_stats(self._h, C.byref(st)))
        return st

    # ---- search -----------------------------------------------------------------------------
    def search(self, params=None):
        self._chk(lib().itsx_search(self._h, C.byref(params) if params is not None else None))

    def search_seqs(self, seq, off, params=None):
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.int64)
        self._nseq = len(off) - 1
        self._chk(lib().itsx_search_seqs(self._h, _p(seq), _p(off), len(off) - 1,
                                         C.byref(params) if params is not None else None))

    def search_seqs_stage1(self, seq, off, params=None):
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.int64)
        self._chk(lib().itsx_search_seqs_stage1(self._h, _p(seq), _p(off), len(off) - 1,
                                                C.byref(params) if params is not None else None))

    def search_stage1(self, params=None):
        self._chk(lib().itsx_search_stage1(self._h, C.byref(params) if params is not None else None))

    def search_shard(self, first, n):
        self._chk(lib().itsx_search_shard(self._h, int(first), int(n)))

    def nreported(self, n_samples=1):
        """Reported hits per profile (hmmsearch's domZ); with n_samples > 1 (set_samples) an [n_samples, P] array."""
        out = np.zeros(max(1, len(self.names) * n_samples), np.int32)
        self._chk(lib().itsx_nreported(self._h, _p(out)))
        out = out[:len(self.names) * n_samples]
        return out if n_samples == 1 else out.reshape(n_samples, len(self.names))

    def set_samples(self, sample_of_read, n_samples):
        """Sample id of every resident read (several samples in one pass; classes and domZ stay per sample)."""
        a = np.ascontiguousarray(sample_of_read, dtype=np.int32)
        self._chk(lib().itsx_reads_set_samples(self._h, _p(a), int(n_samples)))

    def nreported_set(self, arr):
        arr = np.ascontiguousarray(arr, dtype=np.int32)
        self._chk(lib().itsx_nreported_set(self._h, _p(arr)))

    def search_stage2(self):
        self._chk(lib().itsx_search_stage2(self._h))

    def search_stats(self):
        st = SearchStats()
        self._chk(lib().itsx_search_get_stats(self._h, C.byref(st)))
        return st

    def hits(self):
        n = C.c_int64()
        self._chk(lib().itsx_hits(self._h, None, 0, C.byref(n)))
        rows = np.zeros(n.value, dtype=ROW_DTYPE)
        if n.value:
            self._chk(lib().itsx_hits(self._h, _p(rows), n.value, C.byref(n)))
        return rows

    def positions(self, n):
        names = ["start", "stop", "tlen", "left_score10", "left_from", "left_to", "right_score10", "right_from",
                 "right_to"]
        out = {k: np.empty(n, np.int32) for k in names}
        self._chk(lib().itsx_positions(self._h, *[_p(out[k]) for k in names]))
        return out

    def positions_set(self, start, stop, tlen):
        start, stop, tlen = (np.ascontiguousarray(a, dtype=np.int32) for a in (start, stop, tlen))
        self._chk(lib().itsx_positions_set(self._h, _p(start), _p(stop), _p(tlen), len(start)))

    # ---- trim -------------------------------------------------------------------------------
    def trim_set_map(self, uid, n_unique):
        """Install a read -> unique map (uid[i] = -1: read is not in the map and is dropped)."""
        uid = np.ascontiguousarray(uid, dtype=np.int32)
        self._chk(lib().itsx_trim_set_map(self._h, _p(uid), len(uid), int(n_unique)))

    def trim_bounds(self, nreads, mode=0, off_other=None):
        keep = np.empty(nreads, np.uint8)
        lo = np.empty(nreads, np.int32)
        hi = np.empty(nreads, np.int32)
        nk = C.c_int64()
        o = None if off_other is None else np.ascontiguousarray(off_other, dtype=np.int64)
        self._chk(lib().itsx_trim_bounds(self._h, mode, _p(o), nreads, _p(keep), _p(lo), _p(hi), C.byref(nk)))
        return keep, lo, hi, int(nk.value)

    def trim_gather(self, nreads, mode=0, seq=None, qual=None, off=None):
        """Returns (kept_index, out_off, out_seq, out_qual) with the slices packed back to back; out_qual is None
        without qual."""
        nk, tot = C.c_int64(), C.c_int64()
        seq = None if seq is None else np.ascontiguousarray(seq, dtype=np.uint8)
        qual = None if qual is None else np.ascontiguousarray(qual, dtype=np.uint8)
        off = None if off is None else np.ascontiguousarray(off, dtype=np.int64)
        L = lib()
        self._chk(L.itsx_trim_gather(self._h, mode, _p(seq), _p(qual), _p(off), nreads, C.byref(nk), C.byref(tot)))
        ki = np.empty(nk.value, np.int32)
        oo = np.empty(nk.value + 1, np.int64)
        os_ = np.empty(tot.value, np.uint8)
        oq = np.empty(tot.value, np.uint8) if qual is not None else None
        self._chk(L.itsx_run_fetch(self._h, None, None, _p(ki), _p(oo), _p(os_), _p(oq)))
        return ki, oo, os_, oq

    # ---- gzip writer ----------------------------------------------------------------------------
    def gzip_compress(self, data):
        """``data`` (bytes-like or uint8 array) as a multi-member gzip stream compressed on the GPU; returns a uint8
        array (a view of the exact length) that file.write() takes as it is."""
        a = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, np.uint8)
        L = lib()
        cap = int(L.itsx_gzip_bound(a.size))
        out = np.empty(cap, np.uint8)
        n = C.c_int64()
        self._chk(L.itsx_gzip_compress(self._h, _p(a) if a.size else None, a.size, _p(out), cap, C.byref(n)))
        return out[:n.value]

    # ---- paired-end merge -----------------------------------------------------------------------
    def merge_pairs(self, fseq, fqual, foff, rseq, rqual, roff, params=None, fetch=True):
        """Merge R1/R2 records on the GPU.  Returns (merged_len[n], reason[n], merged_index, out_off, out_seq,
        out_qual): the merged reads in input order, packed back to back (the last four are None with fetch=False)."""
        a = [np.ascontiguousarray(x, dtype=np.uint8) for x in (fseq, fqual, rseq, rqual)]
        foff = np.ascontiguousarray(foff, dtype=np.int64)
        roff = np.ascontiguousarray(roff, dtype=np.int64)
        n = len(foff) - 1
        if len(roff) - 1 != n:
            raise ValueError("R1 and R2 hold different numbers of records")
        mlen = np.zeros(n, np.int32)
        reason = np.zeros(n, np.uint8)
        nm, tot = C.c_int64(), C.c_int64()
        L = lib()
        self._chk(L.itsx_merge_pairs(self._h, _p(a[0]), _p(a[1]), _p(foff), _p(a[2]), _p(a[3]), _p(roff), n,
                                     C.byref(params) if params is not None else None, _p(mlen), _p(reason),
                                     C.byref(nm), C.byref(tot)))
        if not fetch:
            return mlen, reason, None, None, None, None
        idx = np.empty(nm.value, np.int32)
        oo = np.zeros(nm.value + 1, np.int64)
        os_ = np.empty(tot.value, np.uint8)
        oq = np.empty(tot.value, np.uint8)
        self._chk(L.itsx_merge_fetch(self._h, _p(idx), _p(oo), _p(os_), _p(oq)))
        return mlen, reason, idx, oo, os_, oq

    def merge_stats(self):
        st = MergeStats()
        self._chk(lib().itsx_merge_get_stats(self._h, C.byref(st)))
        return st

    # ---- whole path ---------------------------------------------------------------------------
    def run(self, seq, off, params=None, out=None):
        """derep + search + positions + single-end trim bounds from host buffers."""
        off = np.ascontiguousarray(off, dtype=np.int64)
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        n = len(off) - 1
        if out is None:
            out = dict(rep=np.empty(n, np.int32), keep=np.empty(n, np.uint8), lo=np.empty(n, np.int32),
                       hi=np.empty(n, np.int32))
        st = RunStats()
        self._chk(lib().itsx_run(self._h, _p(seq), _p(off), n, C.byref(params) if params is not None else None,
                                 _p(out["rep"]), _p(out["keep"]), _p(out["lo"]), _p(out["hi"]), C.byref(st)))
        return out, st

    def reads_upload(self, seq, off):
        off = np.ascontiguousarray(off, dtype=np.int64)
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        self._chk(lib().itsx_reads_upload(self._h, _p(seq), _p(off), len(off) - 1))

    def reads_begin(self, nreads_hint=0, bases_hint=0):
        self._chk(lib().itsx_reads_begin(self._h, int(nreads_hint), int(bases_hint)))

    def reads_append(self, seq, qual, off):
        off = np.ascontiguousarray(off, dtype=np.int64)
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        qual = None if qual is None else np.ascontiguousarray(qual, dtype=np.uint8)
        self._chk(lib().itsx_reads_append(self._h, _p(seq), _p(qual), _p(off), len(off) - 1))

    def reads_end(self):
        n, tb = C.c_int64(), C.c_int64()
        self._chk(lib().itsx_reads_end(self._h, C.byref(n), C.byref(tb)))
        return int(n.value), int(tb.value)

    def trim_gather_range(self, first, count, nbases, mode=0):
        """(kept_index relative to first, out_off, out_seq, out_qual) of the resident reads [first, first + count);
        nbases = bases of the range (worst-case output size)."""
        self._chk(lib().itsx_trim_gather_range(self._h, mode, int(first), int(count), None, None))
        return self.run_fetch(dict(kept_index=np.empty(count, np.int32), out_off=np.empty(count + 1, np.int64),
                                   out_seq=np.empty(nbases, np.uint8), out_qual=np.empty(nbases, np.uint8)))

    def quals_upload(self, qual):
        qual = np.ascontiguousarray(qual, dtype=np.uint8)
        self._chk(lib().itsx_quals_upload(self._h, _p(qual)))

    def derep_resident(self, build_search_set=True):
        nu = C.c_int64()
        self._chk(lib().itsx_derep_resident(self._h, int(bool(build_search_set)), C.byref(nu)))
        return int(nu.value)

    def run_trim(self, seq, qual, off, params=None, out=None):
        """The whole path for one single-end sample, host buffers in and out: derep + search + positions + trim with
        re-expansion.  Returns (dict(kept_index, out_off, out_seq, out_qual[, rep]) trimmed to size, RunStats)."""
        off = np.ascontiguousarray(off, dtype=np.int64)
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        qual = np.ascontiguousarray(qual, dtype=np.uint8)
        n = len(off) - 1
        if out is None:
            out = dict(rep=np.empty(n, np.int32), kept_index=np.empty(n, np.int32), out_off=np.empty(n + 1, np.int64),
                       out_seq=np.empty(len(seq), np.uint8), out_qual=np.empty(len(seq), np.uint8))
        st = RunStats()
        self._chk(lib().itsx_run_trim(self._h, _p(seq), _p(qual), _p(off), n,
                                      C.byref(params) if params is not None else None, _p(out.get("rep")),
                                      _p(out["kept_index"]), _p(out["out_off"]), _p(out["out_seq"]), _p(out["out_qual"]),
                                      C.byref(st)))
        nk, tot = int(st.n_kept), int(st.out_bytes)
        view = dict(kept_index=out["kept_index"][:nk], out_off=out["out_off"][:nk + 1], out_seq=out["out_seq"][:tot],
                    out_qual=out["out_qual"][:tot])
        if out.get("rep") is not None:
            view["rep"] = out["rep"]
        return view, st

    def trim_gather_resident(self, mode=0):
        """Bounds + re-expansion of the resident reads (and qualities), results left on the device -> (n_kept, total)."""
        nk, tot = C.c_int64(), C.c_int64()
        self._chk(lib().itsx_trim_gather_resident(self._h, mode, C.byref(nk), C.byref(tot)))
        return int(nk.value), int(tot.value)

    def run_fetch(self, out=None):
        """Gathered slices left on the device by run_resident() / trim_gather_resident() / trim_gather_range().  out:
        preallocated (pinned) arrays kept_index / out_off / out_seq / out_qual of worst-case size; the returned views
        are cut to size."""
        nk, tot = C.c_int64(), C.c_int64()
        L = lib()
        if out is None:
            self._chk(L.itsx_run_fetch(self._h, C.byref(nk), C.byref(tot), None, None, None, None))
            out = dict(kept_index=np.empty(nk.value, np.int32), out_off=np.empty(nk.value + 1, np.int64),
                       out_seq=np.empty(tot.value, np.uint8), out_qual=np.empty(tot.value, np.uint8))
        self._chk(L.itsx_run_fetch(self._h, C.byref(nk), C.byref(tot), _p(out["kept_index"]), _p(out["out_off"]),
                                   _p(out["out_seq"]), _p(out["out_qual"])))
        return (out["kept_index"][:nk.value], out["out_off"][:nk.value + 1], out["out_seq"][:tot.value],
                out["out_qual"][:tot.value])

    def run_resident(self, params=None):
        st = RunStats()
        self._chk(lib().itsx_run_resident(self._h, C.byref(params) if params is not None else None, C.byref(st)))
        return st
