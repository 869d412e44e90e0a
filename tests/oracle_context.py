"""TEST INFRASTRUCTURE: a stand-in for itsxpress_b200._lib.Context whose compute is the CPU oracle.

The product has no CPU path (a missing CUDA extension or device is an error); this class exists so that the HOST logic
above the C ABI -- the command line, SeqSample / ItsPosition / Dedup, the FASTQ readers and writers, the temp-file policy,
streaming -- can be driven end to end by `-m "not gpu"` tests.  It implements the methods those flows call, with the same
argument meaning and the same array layouts as the ctypes wrapper (itsxpress_b200/_lib.py); tests install it by
monkeypatching `itsxpress_b200.SeqSample.get_context`.  Covered: single-end flows (whole file and streamed) and the
paired flows of one sample (merge, merged and unmerged output), and the batched pass of several samples (classes and
domZ per sample).
"""
import types

import numpy as np

from itsxpress_b200 import _lib


class OracleContext:
    def __init__(self, oracle):
        self.O = oracle
        self.names = []
        self.db = None
        self.side = None
        self.calls = []                       # method names in call order (tests look at the flow taken)
        self._seq = self._off = self._qual = None
        self._parts = None
        self._uid = self._first = None
        self._pos = None
        self._map = None
        self._sample, self._nsamples = None, 1

    def _note(self, name):
        self.calls.append(name)

    # ---- profiles ----
    def load_profiles(self, paths, prefixes=None, skip_missing=True):
        self._note("load_profiles")
        if isinstance(paths, (str, bytes)):
            paths = [paths]
        self.db = self.O.ProfileDB(list(paths), prefixes)
        self.names = list(self.db.names)
        self.side = np.full(len(self.names), -1, np.int8)
        return self.db.n

    def profile_M(self, p):
        return self.db.M[p]

    def set_sides(self, side):
        self.side = np.ascontiguousarray(side, dtype=np.int8)

    def set_sides_by_prefix(self, left_prefix, right_prefix):
        side = np.full(len(self.names), -1, np.int8)
        for i, nm in enumerate(self.names):
            if nm.startswith(left_prefix):
                side[i] = 0
            elif nm.startswith(right_prefix):
                side[i] = 1
        self.set_sides(side)
        return side

    # ---- paired-end merge ----
    def merge_pairs(self, fseq, fqual, foff, rseq, rqual, roff, params=None, fetch=True):
        self._note("merge_pairs")
        foff = np.ascontiguousarray(foff, dtype=np.int64)
        roff = np.ascontiguousarray(roff, dtype=np.int64)
        if len(foff) != len(roff):
            raise ValueError("R1 and R2 hold different numbers of records")
        prm = self.O.merge_params()
        if params is not None:
            for k in ("maxdiffs", "allow_stagger", "qmax", "minovlen", "qmaxout", "qminout", "ascii", "maxee", "maxdiffpct"):
                setattr(prm, k, getattr(params, k))
        mlen, reason, slot_seq, slot_qual = self.O.merge_pairs(fseq, fqual, foff, rseq, rqual, roff, prm)
        idx = np.flatnonzero(reason == 0).astype(np.int32)
        oo = np.zeros(len(idx) + 1, np.int64)
        np.cumsum(mlen[idx], out=oo[1:])
        src = np.repeat((foff[:-1] + roff[:-1])[idx] - oo[:-1], mlen[idx]) + np.arange(int(oo[-1]), dtype=np.int64)
        self._merge = (len(mlen), len(idx), np.bincount(reason, minlength=16))
        if not fetch:
            return mlen, reason, None, None, None, None
        return mlen, reason, idx, oo, slot_seq[src], slot_qual[src]

    def merge_stats(self):
        n, m, by = self._merge
        return types.SimpleNamespace(n_pairs=n, n_merged=m, by_reason=[int(v) for v in by], ms_kernel=0.0, bytes_in=0, bytes_out=0)

    # ---- derep ----
    def _derep(self):
        if self._sample is None:
            rep, strand, nu = self.O.derep(self._seq, self._off)
        else:
            # several samples in one pass: classes never span samples (itsx_reads_set_samples)
            n = len(self._off) - 1
            rep, strand = np.arange(n, dtype=np.int32), np.zeros(n, np.uint8)
            for k in range(self._nsamples):
                idx = np.flatnonzero(self._sample == k)
                if not len(idx):
                    continue
                parts = [self._seq[self._off[i]:self._off[i + 1]] for i in idx]
                o = np.zeros(len(idx) + 1, np.int64)
                o[1:] = np.cumsum([len(p) for p in parts])
                r, st, _ = self.O.derep(np.concatenate(parts), o)
                rep[idx], strand[idx] = idx[r], st
            nu = int(np.count_nonzero(rep == np.arange(n)))
        self._rep, self._strand = rep, strand
        self._first = np.flatnonzero(rep == np.arange(len(rep))).astype(np.int32)
        self._uid = np.searchsorted(self._first, rep).astype(np.int32)
        assert len(self._first) == nu
        return nu

    def reads_upload(self, seq, off):
        self._note("reads_upload")
        self._seq = np.array(seq, dtype=np.uint8)
        self._off = np.array(off, dtype=np.int64)
        self._qual, self._sample = None, None

    def set_samples(self, sample_of_read, n_samples):
        self._sample, self._nsamples = np.array(sample_of_read, dtype=np.int32), int(n_samples)

    def quals_upload(self, qual):
        self._qual = np.array(qual, dtype=np.uint8)
        assert len(self._qual) == len(self._seq)

    def derep_map(self, n):
        assert n == len(self._rep)
        return self._rep.copy(), self._strand.copy(), self._uid.copy()

    def trim_gather_resident(self, mode=0):
        self._note("trim_gather_resident")
        keep, lo, hi = self.O.trim_bounds(self._off, self._uid, self._pos["start"], self._pos["stop"], self._pos["tlen"], mode=mode)
        self._fetch = self._gather(keep, lo, hi, self._seq, self._qual, self._off)
        return len(self._fetch[0]), int(self._fetch[1][-1])

    def run_fetch(self, out=None):
        return self._fetch

    def derep(self, seq, off):
        self._note("derep")
        self._sample = None
        self._seq = np.ascontiguousarray(seq, dtype=np.uint8)
        self._off = np.ascontiguousarray(off, dtype=np.int64)
        self._qual = None
        nu = self._derep()
        return self._rep.copy(), self._strand.copy(), nu

    def derep_clusters(self, n_unique):
        assert n_unique == len(self._first)
        return self._first.copy(), np.bincount(self._uid, minlength=n_unique).astype(np.int32)

    def derep_stats(self):
        return types.SimpleNamespace(ms_total=0.0)

    # ---- streamed ingest ----
    def reads_begin(self, nreads_hint=0, bases_hint=0):
        self._note("reads_begin")
        self._parts = []
        self._sample = None

    def reads_append(self, seq, qual, off):
        self._note("reads_append")
        off = np.ascontiguousarray(off, dtype=np.int64)
        assert off[0] == 0 and len(seq) == off[-1] and (qual is None or len(qual) == len(seq))
        self._parts.append((np.array(seq, np.uint8), None if qual is None else np.array(qual, np.uint8), off.copy()))

    def reads_end(self):
        self._note("reads_end")
        self._seq = np.concatenate([p[0] for p in self._parts]) if self._parts else np.zeros(0, np.uint8)
        self._qual = np.concatenate([p[1] for p in self._parts]) if self._parts else np.zeros(0, np.uint8)
        offs, base = [np.zeros(1, np.int64)], 0
        for p in self._parts:
            offs.append(p[2][1:] + base)
            base += int(p[2][-1])
        self._off = np.concatenate(offs)
        self._parts = None
        return len(self._off) - 1, int(self._off[-1])

    def derep_resident(self, build_search_set=True):
        self._note("derep_resident")
        return self._derep()

    # ---- search ----
    def _run_search(self, seq, off, params):
        prm = self.O.default_params(0, 1)
        if params is not None:
            prm.T, prm.F1, prm.F2, prm.F3, prm.domE = params.T, params.F1, params.F2, params.F3, params.domE
            prm.resolve_multidomain = params.resolve_multidomain
        self._seqlen = np.diff(off).astype(np.int32)
        rows, nrep, _ = self.db.search(self.O.digitize(seq.tobytes()), off, prm)
        self._orows, self._nrep = rows, nrep
        self.search_stage2()

    def search(self, params=None):
        """the resident uniques, first-occurrence order; with several samples resident every sample is searched on its own
        (its own domZ), the positions are those of all uniques in resident order"""
        self._note("search")
        parts = [self._seq[self._off[i]:self._off[i + 1]] for i in self._first]
        uoff = np.zeros(len(parts) + 1, np.int64)
        uoff[1:] = np.cumsum([len(p) for p in parts])
        if self._sample is None:
            self._run_search(np.concatenate(parts) if parts else np.zeros(0, np.uint8), uoff, params)
        else:
            names = ["start", "stop", "tlen", "left_score10", "left_from", "left_to", "right_score10", "right_from", "right_to"]
            pos = {k: np.full(len(parts), -1, np.int32) for k in names}
            of_unique = self._sample[self._first]
            for k in range(self._nsamples):
                u = np.flatnonzero(of_unique == k)
                if not len(u):
                    continue
                o = np.zeros(len(u) + 1, np.int64)
                o[1:] = np.cumsum([len(parts[i]) for i in u])
                self._run_search(np.concatenate([parts[i] for i in u]), o, params)
                for name in names:
                    pos[name][u] = self._pos[name]
            self._pos, self._seqlen = pos, np.diff(uoff).astype(np.int32)
        self._map = (self._uid, None)          # the resident derep map feeds the trim (trim_gather_range)

    def search_seqs(self, seq, off, params=None):
        self._note("search_seqs")
        self._run_search(np.ascontiguousarray(seq, np.uint8), np.ascontiguousarray(off, np.int64), params)

    def search_stage2(self):
        r = self._orows
        self._pos = self.O.itspos(r[r["is_reported"] != 0], self.side, self._seqlen)

    def nreported(self, n_samples=1):
        return self._nrep.astype(np.int32)

    def search_stats(self):
        return types.SimpleNamespace(n_domains_reported=int(np.count_nonzero(self._orows["is_reported"])), ms_total=0.0,
                                     n_selected_multidomain=0)

    def hits(self):
        r = self._orows[self._orows["is_reported"] != 0]
        rows = np.zeros(len(r), dtype=_lib.ROW_DTYPE)
        for k in ("seq", "prof", "ienv", "jenv", "dom_idx", "bitscore", "envsc", "domcorrection", "lnP", "is_multidomain"):
            rows[k] = r[k]
        rows["tlen"] = self._seqlen[r["seq"]]
        rows["seq_score"] = r["bitscore"]       # (full-sequence columns are not what ItsPosition reads)
        rows["seq_lnP"] = r["lnP"]
        rows["reported"] = 1
        return rows

    def positions(self, n):
        assert n == len(self._seqlen)
        return {k: v.copy() for k, v in self._pos.items()}

    # ---- trim ----
    def positions_set(self, start, stop, tlen):
        self._note("positions_set")
        self._table = tuple(np.ascontiguousarray(a, dtype=np.int32) for a in (start, stop, tlen))

    def trim_set_map(self, uid, n_unique):
        self._note("trim_set_map")
        self._map = (np.ascontiguousarray(uid, dtype=np.int32), int(n_unique))

    @staticmethod
    def _gather(keep, lo, hi, seq, qual, off, base=0):
        ki = np.flatnonzero(keep).astype(np.int32)
        lens = (hi - lo)[ki].astype(np.int64)
        oo = np.zeros(len(ki) + 1, np.int64)
        np.cumsum(lens, out=oo[1:])
        idx = np.repeat(off[ki + base] + lo[ki] - oo[:-1], lens) + np.arange(int(oo[-1]), dtype=np.int64)
        return ki, oo, seq[idx], None if qual is None else qual[idx]

    def trim_gather(self, nreads, mode=0, seq=None, qual=None, off=None):
        self._note("trim_gather")
        off = np.ascontiguousarray(off, dtype=np.int64)
        assert nreads == len(off) - 1 == len(self._map[0])
        start, stop, tlen = self._table
        keep, lo, hi = self.O.trim_bounds(off, self._map[0], start, stop, tlen, mode=mode, off_r2=off)
        return self._gather(keep, lo, hi, np.asarray(seq, np.uint8), None if qual is None else np.asarray(qual, np.uint8), off)

    def trim_gather_range(self, first, count, nbases, mode=0):
        """resident reads [first, first + count) through the resident map and the positions of the last search"""
        self._note("trim_gather_range")
        off = self._off[first:first + count + 1]
        assert int(off[-1] - off[0]) == nbases
        keep, lo, hi = self.O.trim_bounds(off - off[0], self._uid[first:first + count], self._pos["start"], self._pos["stop"],
                                          self._pos["tlen"], mode=mode)
        return self._gather(keep, lo, hi, self._seq, self._qual, self._off, base=first)
