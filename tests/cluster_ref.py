"""ctypes binding of tests/cluster_ref.c (the CPU reference of itsx_cluster), and a CPU stand-in context that clusters with
it, so that the command-line tests of clustering also run without a GPU.  The C file is compiled on first use into a
temporary directory (the tree may be read-only)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from itsxpress_b200 import _lib
from oracle_context import OracleContext

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        out = os.path.join(tempfile.mkdtemp(prefix="cluster_ref_"), "libcluster_ref.so")
        cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
        subprocess.check_call([cc, "-O2", "-shared", "-fPIC", "-std=gnu11", "-o", out, os.path.join(_HERE, "cluster_ref.c")])
        L = C.CDLL(out)
        vp = C.c_void_p
        L.ref_cluster.restype = C.c_int64
        L.ref_cluster.argtypes = [vp, vp, vp, C.c_int64, vp, vp, C.c_int32, vp, vp, vp, vp]
        L.ref_accepted_pairs.restype = C.c_int64
        L.ref_accepted_pairs.argtypes = [vp, vp, vp, C.c_int64, vp, vp, C.c_int32, C.c_int64, C.c_int64]
        L.ref_ed.restype = C.c_int
        L.ref_ed.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def default_order(rep):
    """unique indices by abundance descending, then first occurrence (itsx_cluster's order when none is given)"""
    rep = np.asarray(rep)
    first = np.flatnonzero(rep == np.arange(len(rep)))
    ab = np.bincount(np.searchsorted(first, rep), minlength=len(first))
    return np.lexsort((np.arange(len(first)), -ab)).astype(np.int32)


def cluster(seq, off, first, order, cluster_id):
    """(n_centroids, centroid_row_of_unique, strand_of_unique, ed_of_unique, unique_of_row) by brute force"""
    seq = np.ascontiguousarray(seq, np.uint8)
    off = np.ascontiguousarray(off, np.int64)
    first = np.ascontiguousarray(first, np.int32)
    order = np.ascontiguousarray(order, np.int32)
    nu = len(first)
    lens = (off[first + 1] - off[first]) if nu else np.zeros(1, np.int64)
    D = _lib.cluster_dtable(cluster_id, int(lens.max()) if nu else 0)
    crow, strand = np.empty(nu, np.int32), np.empty(nu, np.uint8)
    ed, uor = np.empty(nu, np.int32), np.empty(max(nu, 1), np.int32)
    nc = lib().ref_cluster(_p(seq), _p(off), _p(first), nu, _p(order), _p(D), len(D) - 1, _p(crow), _p(strand), _p(ed),
                           _p(uor))
    return int(nc), crow, strand, ed, uor[:nc]


def accepted_pairs(seq, off, first, cluster_id, group=None):
    """number of unordered pairs of distinct uniques of the same group (per unique; None: one group) whose ed on either
    strand is at most D(max length): the n_accepted of itsx_cluster on these uniques"""
    seq = np.ascontiguousarray(seq, np.uint8)
    off = np.ascontiguousarray(off, np.int64)
    first = np.ascontiguousarray(first, np.int32)
    nu = len(first)
    group = np.zeros(nu, np.int32) if group is None else np.ascontiguousarray(group, np.int32)
    assert len(group) == nu
    lens = (off[first + 1] - off[first]) if nu else np.zeros(1, np.int64)
    D = _lib.cluster_dtable(cluster_id, int(lens.max()) if nu else 0)
    f = lib().ref_accepted_pairs
    if nu < 256:
        return int(f(_p(seq), _p(off), _p(first), nu, _p(group), _p(D), len(D) - 1, 0, nu))
    # chunks of the outer loop on threads (ctypes releases the GIL); small chunks even out the triangle
    import concurrent.futures as cf
    step = max(1, nu // 256)
    with cf.ThreadPoolExecutor(os.cpu_count()) as ex:
        parts = ex.map(lambda a: f(_p(seq), _p(off), _p(first), nu, _p(group), _p(D), len(D) - 1, a, a + step),
                       range(0, nu, step))
        return int(sum(parts))


def ed(a, b, d, rc=False):
    """ed(a, b), or ed(rc(a), b) with rc, if at most d, else d + 1"""
    return lib().ref_ed(a, len(a), b, len(b), d, int(rc))


class ClusterOracleContext(OracleContext):
    """OracleContext that also clusters (with the reference above): afterwards the search set is the centroids and the
    read -> row map points at centroid rows, as on the device."""

    def cluster(self, cluster_id, order=None):
        self._note("cluster")
        if order is None:
            order = default_order(self._rep)
        nc, crow, strand, ed_, uor = cluster(self._seq, self._off, self._first, order, cluster_id)
        self._cl = (crow, strand, ed_, uor)
        self._uid = crow[self._uid] if len(self._uid) else self._uid
        self._first = self._first[uor]
        return nc

    def cluster_fetch(self, n_unique, n_centroids):
        crow, strand, ed_, uor = self._cl
        assert len(crow) == n_unique and len(uor) == n_centroids
        return crow.copy(), strand.copy(), ed_.copy(), uor.copy()

    def cluster_stats(self):
        import types
        return types.SimpleNamespace(n_candidates=0, n_verified=0, n_accepted=0, n_rounds=0, ms_total=0.0)
