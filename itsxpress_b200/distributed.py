"""One sample sharded over the G GPUs of a box (one process per GPU, torch.distributed for the plumbing).

The reference runs one vsearch and one hmmsearch process per sample (itsxpress/SeqSample.py:106-116,
191-209); both are global operations (first occurrence of a class; hmmsearch's per-profile domZ), so a
sharded run needs exactly three exchanges (SURVEY.md 8e):

  1. dereplication, hash-partitioned.  Reads are block-partitioned in input order.  Every rank dereplicates
     its block exactly; each LOCAL unique goes to the owner rank  key64 % G  as one 8-byte record
     (global read index | length << 32) plus its bases: two all-to-alls (records, bases) after one exchange of
     the split sizes.  all_to_all delivers in source-rank order and blocks are contiguous, so the arrival
     order IS ascending global read index: the owner's exact derep of what it received (every class verified
     base by base again) picks the global first occurrence without any sort.
  2. profile search.  The owner searches the classes it owns with the profiles replicated; the per-profile
     count of reported hits -- hmmsearch's domZ -- is all-reduced between stage 1 (scores, -T) and stage 2
     (domE, ItsPosition arg-max).  The same all-reduce carries the number of classes per owner.  An owner decides
     in stage 1 which rows are printed whatever domZ turns out to be (the compact row mode); that needs a bound of
     domZ over the whole sample, the sample's read count, which the split-size exchange of step 1 also carries (one
     more column: every rank's block read count).
  3. answers.  One 16-byte record {representative's global index | strand << 31, start, stop, tlen} per received
     record returns through the inverse all-to-all; the block's position table (one row per local unique) is
     filled from it and the block is trimmed where it lies.  Rank order = input order.  No global table exists.

`run_sharded` is the one orchestration; the compute engine is duck-typed: `GpuEngine` (libitsx_b200 through device
pointers, csrc/shard.cu -- the product; buffers are torch CUDA tensors, collectives are NCCL over NVLink) and, in
the CPU tests, an oracle-backed engine on numpy buffers over gloo (tests/dist_worker.py).
"""
import time

import numpy as np

PHASES = ("local_derep", "plan_pack", "exchange", "owner_derep", "search_stage1", "domz_allreduce", "search_stage2",
          "answers", "answers_exchange", "apply_trim")


# ---- communication ---------------------------------------------------------------------------------------
class Comm:
    """Variable-size exchanges over torch.distributed.  Buffers are torch tensors on `device` (nccl: the rank's GPU)
    or numpy arrays (staged through `device`; gloo: CPU) -- what comes back has the kind that went in."""

    def __init__(self, group=None, device=None):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.group = torch, dist, group
        self.on = dist.is_available() and dist.is_initialized()
        self.rank = dist.get_rank(group) if self.on else 0
        self.world = dist.get_world_size(group) if self.on else 1
        backend = dist.get_backend(group) if self.on else "none"
        self.device = device if device is not None else (
            torch.device("cuda", torch.cuda.current_device()) if backend == "nccl" else torch.device("cpu"))
        self.cuda = self.device.type == "cuda"
        self.bytes_sent = {}           # collective name -> bytes this rank put on the wire (excluding its own share)

    def _t(self, a):
        if isinstance(a, np.ndarray):
            return self.torch.from_numpy(np.ascontiguousarray(a)).to(self.device)
        return a.contiguous()

    def _back(self, t, like):
        return t.cpu().numpy() if isinstance(like, np.ndarray) else t

    def sync(self):
        if self.cuda:
            self.torch.cuda.current_stream(self.device).synchronize()

    def exchange_counts(self, counts):
        """counts: int64 [G, k] (row g goes to rank g) -> int64 [G, k] (row g came from rank g), numpy."""
        counts = np.ascontiguousarray(counts, np.int64)
        if self.world == 1:
            return counts.copy()
        t = self._t(counts.reshape(-1))
        out = self.torch.empty_like(t)
        self.dist.all_to_all_single(out, t, group=self.group)
        return out.cpu().numpy().reshape(counts.shape)

    def all_to_all(self, x, send, recv, name=None):
        """x: 1-D or [n, k] buffer laid out by destination rank; send / recv: rows per rank."""
        send, recv = [int(v) for v in send], [int(v) for v in recv]
        if name is not None:
            row = (x.dtype.itemsize if isinstance(x, np.ndarray) else x.element_size()) * \
                (int(np.prod(x.shape[1:])) if x.ndim > 1 else 1)
            self.bytes_sent[name] = self.bytes_sent.get(name, 0) + row * (sum(send) - send[self.rank])
        if self.world == 1:
            return x.copy() if isinstance(x, np.ndarray) else x.clone()
        t = self._t(x)
        out = self.torch.empty((sum(recv),) + tuple(t.shape[1:]), dtype=t.dtype, device=self.device)
        self.dist.all_to_all_single(out, t, recv, send, group=self.group)
        return self._back(out, x)

    def all_reduce_sum(self, arr):
        arr = np.ascontiguousarray(arr, np.int64)
        if self.world == 1:
            return arr.copy()
        t = self._t(arr)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)
        return t.cpu().numpy()


# ---- the product engine --------------------------------------------------------------------------------------
class GpuEngine:
    """The block side (`local`) and the owner side (`owner`) of a sharded run on libitsx_b200: two contexts on the
    rank's GPU, every exchange buffer a torch CUDA tensor handed to the C ABI by device pointer (no CPU path)."""

    def __init__(self, local, owner, params=None):
        import ctypes as C
        import torch
        from ._lib import lib
        self.C, self.torch, self.L = C, torch, lib()
        self.local, self.owner, self.params = local, owner, params
        self.dev = torch.device("cuda", int(local.device))
        self.n = self.nu = self.m = 0
        self.n_reads_sample = 0
        self.resident = self.resident_qual = False

    def _p(self, t):
        if t is None:
            return None
        if isinstance(t, np.ndarray):
            return t.ctypes.data_as(self.C.c_void_p)
        return self.C.c_void_p(t.data_ptr()) if t.numel() else None

    # -- block side --
    def upload(self, seq, off, qual=None):
        """Make the block resident ahead of the timed region (bench `value`); run_sharded then skips the upload."""
        self.local.reads_upload(seq, off)
        if qual is not None:
            self.local.quals_upload(qual)
        self.n = len(off) - 1
        self.resident = True
        self.resident_qual = qual is not None

    def local_derep(self, seq, off):
        if not self.resident:
            self.local.reads_upload(seq, off)
            self.n = len(off) - 1
        self.nu = self.local.derep_resident(build_search_set=False)
        return self.nu

    def plan(self, G):
        rc, bc = np.zeros(G, np.int64), np.zeros(G, np.int64)
        self.local._chk(self.L.itsx_shard_plan(self.local._h, G, self._p(rc), self._p(bc)))
        return rc, bc

    def pack(self, gidx0, nbytes):
        t = self.torch
        rec = t.empty(self.nu, dtype=t.int64, device=self.dev)
        bases = t.empty(int(nbytes), dtype=t.uint8, device=self.dev)
        self.local._chk(self.L.itsx_shard_pack(self.local._h, int(gidx0), self._p(rec), self._p(bases)))
        return rec, bases

    # -- owner side --
    def owner_derep(self, rec, bases):
        n_own = self.C.c_int64()
        self.m = int(rec.shape[0])
        self.owner._chk(self.L.itsx_shard_owner_derep(self.owner._h, self._p(rec), self.m, self._p(bases),
                                                      int(bases.shape[0]), self.C.byref(n_own)))
        return int(n_own.value)

    def sample_reads(self, n_reads):
        """The sample's read count (run_sharded learns it in the split-size exchange).  It bounds any profile's domZ, so
        params that leave domz_upper at 0 ("this context's sequence count", too small for an owner that searches a
        share of the classes) get it in a copy in search_stage1; an explicit domz_upper is kept."""
        self.n_reads_sample = int(n_reads)

    def search_stage1(self):
        from ._lib import SearchParams, default_params
        prm = default_params() if self.params is None else SearchParams.from_buffer_copy(self.params)
        if prm.domz_upper == 0:
            prm.domz_upper = self.n_reads_sample
        self.owner.search_stage1(prm)
        return self.owner.nreported().astype(np.int64)

    def search_stage2(self, nrep_global):
        self.owner.nreported_set(nrep_global.astype(np.int32))
        self.owner.search_stage2()

    def answers(self):
        t = self.torch
        ans = t.empty((self.m, 4), dtype=t.int32, device=self.dev)
        self.owner._chk(self.L.itsx_shard_answers(self.owner._h, self.m, self._p(ans)))
        return ans

    # -- block side again --
    def apply(self, ans, want_rep=True):
        rep = np.empty(self.n, np.int64) if want_rep else None
        strand = np.empty(self.n, np.uint8) if want_rep else None
        self.local._chk(self.L.itsx_shard_apply(self.local._h, self._p(ans), self.nu, self._p(rep), self._p(strand)))
        return rep, strand

    def trim_bounds(self, mode=0):
        keep, lo, hi, nk = self.local.trim_bounds(self.n, mode=mode)
        return keep, lo, hi

    def trim_gather(self, qual=None, mode=0, out=None, fetch=True):
        """Re-expansion of the block: kept_index, out_off, out_seq, out_qual.  qual: host qualities of the block when they
        are not resident (uploaded here).  out: preallocated (pinned) worst-case arrays for the copy back.  fetch=False:
        the slices stay in HBM (-> (n_kept, total))."""
        if qual is not None:
            self.local.quals_upload(qual)
        nk, tot = self.local.trim_gather_resident(mode)
        if not fetch:
            return nk, tot
        return self.local.run_fetch(out)


# ---- helpers ---------------------------------------------------------------------------------------------------
def block_range(n, rank, world):
    """[lo, hi) of rank's block when n items are dealt in contiguous, near-equal blocks."""
    base, extra = divmod(n, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


# ---- the sharded hot path --------------------------------------------------------------------------------------
def run_sharded(engine, comm, seq, off, first_global_index, phases=None, want_rep=True, gather=False, qual=None,
                gather_out=None):
    """Hot path for this rank's block of one sample.

    seq/off: this rank's reads (ASCII back to back, int64 offsets; ignored by an engine whose block is already
    resident); first_global_index: global index of its first read.  Returns dict(rep=global representative index per
    local read (int64), strand, keep, lo, hi, n_unique_global, n_owned, nreported[, kept_index, out_off, out_seq,
    out_qual with gather=True; gather="device" leaves the slices in HBM and returns only n_kept / out_bytes]).  Results are identical to the single-GPU path on the concatenated input.
    phases: dict that receives the seconds spent per phase (PHASES), accumulated.
    seq/off None: the engine's block is resident and its `n` is the block's read count.
    """
    G = comm.world
    t_last = [time.perf_counter()]

    def lap(name):
        comm.sync()
        now = time.perf_counter()
        if phases is not None:
            phases[name] = phases.get(name, 0.0) + (now - t_last[0])
        t_last[0] = now

    # 1a. exact derep of the block
    nu_l = engine.local_derep(seq, off)
    lap("local_derep")
    # 1b. local uniques -> owner = key % G: bucket, record stream + bases in bucket order
    rec_counts, byte_counts = engine.plan(G)
    rec, bases = engine.pack(first_global_index, int(byte_counts.sum()))
    lap("plan_pack")
    # every rank also sends its block's read count: their sum is the sample's, which bounds any profile's domZ
    n_block = len(off) - 1 if off is not None else engine.n
    got = comm.exchange_counts(np.stack([rec_counts, byte_counts, np.full(G, n_block, np.int64)], axis=1))
    rrc, rbc = got[:, 0], got[:, 1]
    if hasattr(engine, "sample_reads"):        # an engine that bounds domZ in stage 1 (GpuEngine's compact row mode)
        engine.sample_reads(int(got[:, 2].sum()))
    rec_in = comm.all_to_all(rec, rec_counts, rrc, name="records")
    bases_in = comm.all_to_all(bases, byte_counts, rbc, name="bases")
    lap("exchange")
    # 1c. owner: exact derep of the received uniques; arrival order = ascending global read index
    n_own = engine.owner_derep(rec_in, bases_in)
    lap("owner_derep")
    # 2. the owner searches the classes it owns; domZ is global (and so is the class count)
    nrep_local = engine.search_stage1()
    lap("search_stage1")
    red = comm.all_reduce_sum(np.concatenate([nrep_local, [n_own]]).astype(np.int64))
    nrep_global, n_unique_global = red[:-1], int(red[-1])
    lap("domz_allreduce")
    engine.search_stage2(nrep_global)
    lap("search_stage2")
    # 3. answers home through the inverse all-to-all; trim the block where it lies
    ans = engine.answers()
    lap("answers")
    ans_back = comm.all_to_all(ans, rrc, rec_counts, name="answers")
    lap("answers_exchange")
    rep_global, strand = engine.apply(ans_back, want_rep=want_rep)
    out = dict(rep=rep_global, strand=strand, n_unique_global=n_unique_global, n_owned=int(n_own),
               nreported=nrep_global, n_local_unique=int(nu_l))
    if gather == "device":
        nk, tot = engine.trim_gather(qual=qual, fetch=False)
        out.update(n_kept=nk, out_bytes=tot)
    elif gather:
        ki, oo, os_, oq = engine.trim_gather(qual=qual, out=gather_out)
        out.update(kept_index=ki, out_off=oo, out_seq=os_, out_qual=oq, n_kept=len(ki), out_bytes=len(os_))
    else:
        keep, lo, hi = engine.trim_bounds()
        out.update(keep=keep, lo=lo, hi=hi)
    lap("apply_trim")
    return out
