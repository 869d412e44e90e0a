"""Many ranks of one sharded sample in one process, and what their exchanges must look like.

`ThreadComm` implements the `Comm` interface of itsxpress_b200.distributed over threads of this process: the ranks of
one world share a slot table and a barrier, and every collective copies what each rank hands in.  `run_world` runs
the real `run_sharded` on every rank at once (the C library releases the GIL in its calls, so the ranks really do
overlap), so G ranks of the product's sharded path run on ONE GPU -- each rank with its own LOCAL and OWNER context --
and the CPU suite runs the same with the oracle-backed engine.  `derep_ref` is a plain restatement of the
dereplication (derep.cu's header, SURVEY Appendix B); `check_derep` and `check_exchange` hold a world's results and
recorded exchanges to it.
"""
import threading

import numpy as np

from itsxpress_b200.distributed import block_range, run_sharded

_COMP = bytes.maketrans(b"ACGTRYMKHDBV", b"TGCAYRKMDHVB")


# ---- the reference --------------------------------------------------------------------------------------------
def normalise(s):
    """Residues upper-cased, U read as T; every other byte stays."""
    return s.upper().replace(b"U", b"T")


def revcomp(s):
    """Reverse complement of the normalised read: A/T, C/G, R/Y, M/K, H/D, B/V swap, every other byte maps to itself."""
    return normalise(s).translate(_COMP)[::-1]


def derep_ref(reads):
    """Exact dereplication over both strands: a read's class is min(s, revcomp(s)) of its normalised bytes, the
    representative is the class's first read in index order, strand = 0 iff the read equals its representative.
    Returns (rep int64[n], strand uint8[n], number of classes)."""
    first = {}
    rep = np.empty(len(reads), np.int64)
    strand = np.empty(len(reads), np.uint8)
    for i, s in enumerate(reads):
        t = normalise(s)
        r = first.setdefault(min(t, revcomp(s)), i)
        rep[i] = r
        strand[i] = 0 if t == normalise(reads[r]) else 1
    return rep, strand, len(first)


def pack(reads, quals=None):
    """reads (list of bytes) -> (seq uint8, off int64[n + 1]), and the qualities alike."""
    off = np.zeros(len(reads) + 1, np.int64)
    off[1:] = np.cumsum([len(r) for r in reads])
    seq = np.frombuffer(b"".join(reads), np.uint8).copy()
    if quals is None:
        return seq, off
    return seq, off, np.frombuffer(b"".join(quals), np.uint8).copy()


def unpack(seq, off):
    return [seq[off[i]:off[i + 1]].tobytes() for i in range(len(off) - 1)]


# ---- read sets ----------------------------------------------------------------------------------------------------
def rand_reads(rng, n, lo, hi, dup_frac=0.5, rc_frac=0.3, lower_frac=0.1, iupac_frac=0.05, u_frac=0.02):
    """n reads of lo..hi bases; about dup_frac of them repeat an earlier one, on either strand, in either case, some
    with U for T; a few carry an IUPAC symbol or N."""
    base, reads = [], []
    for _ in range(n):
        if base and rng.random() < dup_frac:
            s = base[rng.integers(len(base))]
            if rng.random() < rc_frac:
                s = revcomp(s)
            if rng.random() < lower_frac:
                s = s.lower()
            if rng.random() < u_frac:
                s = s.replace(b"T", b"U").replace(b"t", b"u")
        else:
            L = int(rng.integers(lo, hi + 1))
            s = rng.choice(np.frombuffer(b"ACGT", np.uint8), L).tobytes()
            if L and rng.random() < iupac_frac:
                p = int(rng.integers(L))
                s = s[:p] + bytes([rng.choice(np.frombuffer(b"NRYMKHDBVSW", np.uint8))]) + s[p + 1:]
            base.append(s)
        reads.append(s)
    return reads


def fixture_case(seq, off, qual):
    """The fixture's reads with IUPAC symbols put into three of them, then reverse-complement, lower-case and U copies
    of fixture reads at the end (the last ranks), so that classes with both strands and cases span ranks."""
    reads, quals = unpack(seq, off), unpack(qual, off)
    for i, p, c in ((7, 30, b"R"), (60, 45, b"K"), (130, 12, b"N")):
        reads[i] = reads[i][:p] + c + reads[i][p + 1:]
    extra = [(revcomp(reads[i]), quals[i][::-1]) for i in (3, 7, 50, 60, 101, 150, 200)]
    extra += [(reads[i].lower(), quals[i]) for i in (10, 60, 80, 130, 160)]
    extra += [(revcomp(reads[130]).lower(), quals[130][::-1]), (reads[5].replace(b"T", b"U"), quals[5])]
    return reads + [r for r, _ in extra], quals + [q for _, q in extra]


def spread_revcomp_copies(seq, off, qual, every=7, first=400):
    """Reverse complements of every `every`-th of the first `first` reads, spread evenly over the rest of the sample
    (so classes with both strands span ranks); qualities reversed with them."""
    reads, quals = unpack(seq, off), unpack(qual, off)
    src = list(range(0, min(len(reads), first), every))
    step = max(1, (len(reads) - first) // (len(src) + 1))
    out_r, out_q = reads[:first], quals[:first]
    pos = first
    for i in src:
        out_r += reads[pos:pos + step] + [revcomp(reads[i])]
        out_q += quals[pos:pos + step] + [quals[i][::-1]]
        pos += step
    return out_r + reads[pos:], out_q + quals[pos:]


def degenerate_reads(kind):
    """Edge cases of the sharded derep.  "main": empty reads on several ranks; 1-base reads (A, T, a, U); palindromes;
    lengths 15-17, 31-33 and 63-65 whose reverse complements come later (the owner re-packs their bases at other
    offsets, so the 2-bit words straddle differently); IUPAC / N reads whose first occurrence is the lower-case or the
    reverse-complement form.  "twenty" / "five": 20 and 5 reads of the same kinds (more ranks than reads)."""
    rng = np.random.default_rng(11)

    def rand(L):
        return rng.choice(np.frombuffer(b"ACGT", np.uint8), L).tobytes()

    front, back = [], []
    for L in (15, 16, 17, 31, 32, 33, 63, 64, 65):
        s = rand(L)
        front.append(s)
        back.append(revcomp(s))
    half = rand(16)
    pal, pal33 = half + revcomp(half), rand(33)
    front += [b"A", b"T", b"a", b"U", b"ACGT", b"GAATTC", pal, pal33]
    back += [b"acgt", b"gaattc", pal.lower(), revcomp(pal33).lower(), b"t", b"u"]
    iu1 = rand(10) + b"N" + rand(9) + b"R" + rand(19)
    iu2 = rand(5) + b"Y" + rand(20) + b"KWS" + rand(6) + b"N"
    iu3 = rand(31) + b"B" + rand(1) + b"H"                 # 34 bases, symbols across the 32-base boundary
    front += [iu1.lower(), revcomp(iu2), revcomp(iu3).lower()]
    back += [iu1, revcomp(iu1), iu2.lower(), iu2, iu3, b"NNNN", b"nnnn"]
    if kind == "main":
        return [b""] + front[:9] + [b"", b""] + front[9:] + [b""] + back[:10] + [b""] + back[10:] + [b"", b""]
    if kind == "twenty":
        return ([b"", b"A", front[0], iu1.lower(), pal, b"U", front[5], revcomp(iu2), b""] +
                [b"t", back[0], iu1, b"", back[5], pal.lower(), iu2, b"a", b"NNNN", b"nnnn", b""])
    if kind == "five":
        return [b"", b"ACGT", b"a", b"", b"T"]
    if kind == "empty":
        return [b""] * 6
    raise ValueError(kind)


# ---- ranks as threads -------------------------------------------------------------------------------------------
class ThreadWorld:
    """What the G ranks of one run share: the slot table every collective goes through, the barrier, and a copy of
    every exchanged buffer (`sent[name][rank] = (buffer as numpy, split sizes)`; "counts" holds the split-size table)."""

    def __init__(self, G, timeout=300.0):
        self.G = G
        self.barrier = threading.Barrier(G, timeout=timeout)
        self.slots = [None] * G
        self.sent = {}
        self.lock = threading.Lock()

    def gather(self, rank, value):
        """Every rank's value, in rank order (a collective: all ranks call it)."""
        self.slots[rank] = value
        self.barrier.wait()
        got = list(self.slots)
        self.barrier.wait()             # nobody overwrites a slot before every rank has read them all
        return got

    def record(self, name, rank, buf, send):
        with self.lock:
            self.sent.setdefault(name, [None] * self.G)[rank] = (buf, list(send))


def _as_numpy(x):
    return np.array(x, copy=True) if isinstance(x, np.ndarray) else x.detach().cpu().numpy().copy()


class ThreadComm:
    """`itsxpress_b200.distributed.Comm` for one rank of a ThreadWorld: buffers are numpy arrays or torch tensors (CUDA
    ones stay on the device), what comes back has the kind that went in."""

    def __init__(self, world, rank, device=None):
        self.hub, self.rank, self.world = world, rank, world.G
        self.device = device
        self.cuda = device is not None and getattr(device, "type", None) == "cuda"
        self.bytes_sent = {}

    def sync(self):
        if self.cuda:
            import torch
            torch.cuda.current_stream(self.device).synchronize()

    def exchange_counts(self, counts):
        counts = np.array(counts, np.int64, copy=True)
        self.hub.record("counts", self.rank, counts, [1] * self.world)
        got = self.hub.gather(self.rank, counts)
        return np.stack([got[g][self.rank] for g in range(self.world)])

    def all_to_all(self, x, send, recv, name=None):
        send, recv = [int(v) for v in send], [int(v) for v in recv]
        if name is not None:
            row = (x.dtype.itemsize if isinstance(x, np.ndarray) else x.element_size()) * \
                (int(np.prod(x.shape[1:])) if x.ndim > 1 else 1)
            self.bytes_sent[name] = self.bytes_sent.get(name, 0) + row * (sum(send) - send[self.rank])
            self.hub.record(name, self.rank, _as_numpy(x), send)
        assert len(send) == len(recv) == self.world and sum(send) == x.shape[0]
        got = self.hub.gather(self.rank, (x, send))
        pieces = []
        for src, (xs, ss) in enumerate(got):            # source-rank order
            a = sum(ss[:self.rank])
            assert ss[self.rank] == recv[src], ("split sizes disagree", src, self.rank, ss[self.rank], recv[src])
            pieces.append(xs[a:a + ss[self.rank]])
        if isinstance(x, np.ndarray):
            return np.concatenate(pieces)
        import torch
        out = torch.cat(pieces)
        if out.is_cuda:
            torch.cuda.current_stream(out.device).synchronize()
        return out

    def all_reduce_sum(self, arr):
        got = self.hub.gather(self.rank, np.array(arr, np.int64, copy=True))
        return np.sum(got, axis=0)


def run_threads(G, fn, timeout=300.0):
    """fn(rank, world) on G threads; returns ([result of every rank], world).  A rank that raises aborts the barrier so
    the others stop waiting; the first exception that is not the resulting BrokenBarrierError is re-raised."""
    world = ThreadWorld(G, timeout)
    res, err = [None] * G, [None] * G

    def body(r):
        try:
            res[r] = fn(r, world)
        except BaseException as e:       # noqa: B902 -- handed to the caller below
            err[r] = e
            world.barrier.abort()

    threads = [threading.Thread(target=body, args=(r,), name="rank%d" % r) for r in range(G)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    errs = [e for e in err if e is not None]
    if errs:
        real = [e for e in errs if not isinstance(e, threading.BrokenBarrierError)]
        raise (real or errs)[0]
    return res, world


def run_world(G, seq, off, make_engine, qual=None, device=None, **kw):
    """run_sharded on G ranks over the contiguous blocks of (seq, off); make_engine(rank) gives each rank's engine.
    Returns ([run_sharded's dict per rank], world, [(lo, hi) per rank])."""
    n = len(off) - 1
    blocks = [block_range(n, r, G) for r in range(G)]

    def rank_fn(r, world):
        lo, hi = blocks[r]
        b0, b1 = int(off[lo]), int(off[hi])
        q = None if qual is None else qual[b0:b1]
        return run_sharded(make_engine(r), ThreadComm(world, r, device), seq[b0:b1], off[lo:hi + 1] - b0, lo,
                           qual=q, **kw)

    outs, world = run_threads(G, rank_fn)
    return outs, world, blocks


# ---- GPU contexts ------------------------------------------------------------------------------------------------
class ContextPool:
    """Contexts on GPU 0, made once and reused by every case (stale state from a previous case is part of what runs):
    LOCAL and OWNER contexts for the largest G used so far, and one context for the single-GPU path."""

    def __init__(self):
        self.local, self.owner, self._single = [], [], None

    def ranks(self, G):
        from itsxpress_b200 import _lib
        while len(self.local) < G:
            pair = _lib.Context(0), _lib.Context(0)
            self.local.append(pair[0])
            self.owner.append(pair[1])
        return self.local[:G], self.owner[:G]

    @property
    def single(self):
        from itsxpress_b200 import _lib
        if self._single is None:
            self._single = _lib.Context(0)
        return self._single

    def close(self):
        for c in self.local + self.owner + ([self._single] if self._single else []):
            c.close()
        self.local, self.owner, self._single = [], [], None


POOL = ContextPool()


def load_profiles(ctxs, paths, prefixes):
    for c in ctxs:
        c.load_profiles(paths, prefixes)
        c.set_sides_by_prefix(*prefixes)


def run_ranks(G, contexts, seq, off, qual=None, params=None, **kw):
    """run_sharded(GpuEngine(local[r], owner[r], params), ThreadComm, ...) on every rank r < G of one GPU."""
    import torch
    from itsxpress_b200.distributed import GpuEngine
    local, owner = contexts
    return run_world(G, seq, off, lambda r: GpuEngine(local[r], owner[r], params), qual=qual,
                     device=torch.device("cuda", 0), **kw)


# ---- checks --------------------------------------------------------------------------------------------------------
def check_derep(outs, blocks, reads, ref=None):
    """(a) Global representative, strand, class count and Σ n_owned of every rank against derep_ref."""
    rep, strand, nu = ref if ref is not None else derep_ref(reads)
    for o, (lo, hi) in zip(outs, blocks):
        assert np.array_equal(np.asarray(o["rep"], np.int64), rep[lo:hi]), ("rep", lo, hi)
        assert np.array_equal(np.asarray(o["strand"], np.uint8), strand[lo:hi]), ("strand", lo, hi)
        assert o["n_unique_global"] == nu
        assert o["n_local_unique"] == derep_ref(reads[lo:hi])[2]
    assert sum(o["n_owned"] for o in outs) == nu


def _records(buf):
    r = np.asarray(buf).view(np.uint64)
    return (r & np.uint64(0xffffffff)).astype(np.int64), (r >> np.uint64(32)).astype(np.int64)


def check_exchange(world, blocks, reads, ref=None):
    """(b) The exchanges as the ranks sent them.  Returns owner_of_class: global representative -> owning rank."""
    G = world.G
    rep, strand, _ = ref if ref is not None else derep_ref(reads)
    counts, recs, bases, answers = (world.sent[k] for k in ("counts", "records", "bases", "answers"))
    owner_of_class = {}
    arrivals = [[] for _ in range(G)]          # per owner: global indices in arrival order
    for src, (lo, hi) in enumerate(blocks):
        cnt = counts[src][0]
        gidx, glen = _records(recs[src][0])
        rsend, bsend = recs[src][1], bases[src][1]
        assert cnt.shape == (G, 3) and list(cnt[:, 0]) == rsend and list(cnt[:, 1]) == bsend, "split sizes != plan"
        assert np.all(cnt[:, 2] == hi - lo), "block read count"
        assert len(gidx) == sum(rsend) and len(bases[src][0]) == sum(bsend)
        # every local unique exactly once: the block's first occurrences, as global indices
        lrep = derep_ref(reads[lo:hi])[0]
        assert np.array_equal(np.sort(gidx), np.flatnonzero(lrep == np.arange(hi - lo)) + lo), "local uniques"
        b = bases[src][0]
        r0 = 0
        boff = np.concatenate([[0], np.cumsum(glen)])
        for dst in range(G):
            g = gidx[r0:r0 + rsend[dst]]
            assert np.all(np.diff(g) > 0), ("bucket not ascending", src, dst)
            assert int(glen[r0:r0 + rsend[dst]].sum()) == bsend[dst], ("bucket bytes", src, dst)
            for j in range(r0, r0 + rsend[dst]):
                s = reads[gidx[j]]
                assert glen[j] == len(s) and b[boff[j]:boff[j + 1]].tobytes() == s, ("record", src, gidx[j])
                cls = int(rep[gidx[j]])
                assert owner_of_class.setdefault(cls, dst) == dst, ("class split over owners", cls)
            arrivals[dst].append(g)
            r0 += rsend[dst]
    for dst in range(G):
        got = np.concatenate(arrivals[dst]) if arrivals[dst] else np.zeros(0, np.int64)
        assert np.all(np.diff(got) > 0), ("arrivals not ascending", dst)
        # the owner's answers, in arrival order: the class's global representative and the record's strand against it
        ans, asend = answers[dst]
        assert sum(asend) == len(got) == len(ans) and list(asend) == [recs[s][1][dst] for s in range(G)]
        a = np.ascontiguousarray(np.asarray(ans, np.int32).reshape(-1, 4)[:, 0]).view(np.uint32)
        assert np.array_equal((a & np.uint32(0x7fffffff)).astype(np.int64), rep[got]), ("answer rep", dst)
        assert np.array_equal((a >> np.uint32(31)).astype(np.uint8), strand[got]), ("answer strand", dst)
    return owner_of_class
