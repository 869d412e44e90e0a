#!/usr/bin/env python
"""bench.py -- headline benchmark of the ITSxpress hot path on B200.

One "step" = one pass of the whole hot path over one synthetic sample of BASELINE.json configs[1] (1 M single-end
250 bp ITS1 reads, 30 % unique): exact derep -> profile-HMM cascade -> boundary selection -> trim bounds ->
re-expansion (trimmed bases + qualities of every kept read).  F.hmm (Fungi) is missing from the reference mount, so
the largest present analogue M.hmm (Metazoa, 98 ITS1 profiles) stands in -- stated in `config`.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2] [--scale S] [--impl reference] [--replicas]
                  [--dump-outputs DIR]

value  reads/s with the reads (bases, qualities, offsets) resident in HBM when the timed region starts
e2e    reads/s through the C-ABI call with pinned HOST buffers: itsx_run_trim = H2D of bases + qualities + offsets,
       kernels, D2H of the trimmed bases + qualities + offsets (what Dedup.create_trimmed_seqs writes, minus titles)
N = 1  one sample on one GPU.
N > 1  (torchrun, one rank per GPU) THE SAME sample sharded over the ranks -- SURVEY 8e's split: block-partitioned
       reads, hash-partitioned exact derep through an NCCL all-to-all, owners search their classes with the
       profiles replicated, domZ all-reduce, answers through the inverse all-to-all, every rank trims its block.
       Strong scaling; results are checked against the one-GPU path on rank 0 after the timed region.
       --replicas: one independent sample per rank instead (QIIME 2 artifacts; weak scaling, no collective).
--impl reference  times the CPU oracle (restatement of vsearch + hmmsearch + ItsPosition + trim, all host threads) on
       a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import synth  # noqa: E402

INT_OPS_PER_2CELLS = 3.0      # VIMNMX (xB), VIADDMNMX (score, floor), half a VIMNMX3 x2 (row max): one s16x2 MSV cell pair
FP_OPS_PER_CELL = 10.0        # Forward 11 + Backward 9 FMA-pipe instructions per M/I/D cell, averaged
ENV_OPS_PER_CELL = 11.0       # envelope: Forward 11 + Backward 9 + decoding 2 per row cell, counted as 2 cells
# issue rates measured on this pool's B200 with tools/ubench/ffma2.cu (profiles/r1_ubench_issue_rates.txt):
# warp-instructions per clock per SM at 1965 MHz
MEASURED_FFMA_PER_CLK_SM = 3.820
MEASURED_S16X2_PER_CLK_SM = 1.959
NVLINK_GBS = 770.0            # measured peer copy bandwidth per direction per GPU (B200_PROFILING.md)

WORKLOAD_NAMES = {"c2": "BASELINE configs[1]", "c2_small": "configs[1] reduced", "c4s": "configs[3] shape, scaled",
                  "c3s": "configs[2] shape, scaled", "c3": "BASELINE configs[2]", "c4": "BASELINE configs[3]"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    d = {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "source": "fallback"}
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            d.update(hbm_gbs=float(j["hbm_gbs"]), sm_max_mhz=float(j.get("sm_max_mhz", 1965.0)), source="measured")
        except Exception:
            pass
    f = d["sm_max_mhz"] * 1e6
    # cells/s = SMs x warp-instr/clk/SM x 32 lanes x f / instructions per cell
    d["int_gcups"] = 148 * MEASURED_S16X2_PER_CLK_SM * 32 * f * 2.0 / INT_OPS_PER_2CELLS / 1e9
    d["fp_gcups"] = 148 * MEASURED_FFMA_PER_CLK_SM * 32 * f / FP_OPS_PER_CELL / 1e9
    d["env_gcups"] = 148 * MEASURED_FFMA_PER_CLK_SM * 32 * f / ENV_OPS_PER_CELL / 1e9
    return d


def kernel_traffic(kname):
    """DRAM bytes per launch of `kname` from this round's ncu --set full capture at bench scale
    (profiles/traffic.json names the capture it was read from); None when no capture is committed."""
    try:
        j = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        k = j["kernels"][kname]
        return float(k["dram_bytes_per_launch"]), "%s (%s)" % (j["source"], k.get("note", "per launch"))
    except Exception:
        return None, "no ncu capture committed for this kernel"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_sample(seq, off, which, frac_mod=12, pick=7):
    """Bounded sample that keeps the workload's unique fraction: all reads of every 12th unique
    (~80 k reads, ~10 s on 16 cores)."""
    sel = np.flatnonzero((which % frac_mod) == pick)
    lens = (off[1:] - off[:-1])[sel]
    o = np.zeros(len(sel) + 1, np.int64)
    o[1:] = np.cumsum(lens)
    delta = np.repeat(off[sel] - o[:-1], lens)
    s = seq[delta + np.arange(int(o[-1]), dtype=np.int64)]
    return s, o, ("all reads of every %dth unique (%d reads, %d uniques) of the workload; reads/s of the whole workload "
                  "is taken to be the subsample's (the CPU path is linear in reads x profiles)" %
                  (frac_mod, len(sel), len(np.unique(which[sel]))))


def oracle_pipeline(O, db, side, seq, off, threads=0, want_pos=False):
    """derep -> search -> ItsPosition -> trim bounds on the CPU oracle; returns kept count (and the per-read arrays)."""
    rep, strand, nu = O.derep(seq, off)
    idx = np.flatnonzero(rep == np.arange(len(rep)))
    lens = (off[1:] - off[:-1])[idx]
    uoff = np.zeros(len(idx) + 1, np.int64)
    uoff[1:] = np.cumsum(lens)
    delta = np.repeat(off[idx] - uoff[:-1], lens)
    useq = seq[delta + np.arange(int(uoff[-1]), dtype=np.int64)]
    codes = O.digitize(useq.tobytes())
    rows, nrep, st = db.search(codes, uoff, O.default_params(threads))
    pos = O.itspos(rows, side, lens.astype(np.int32))
    n = len(rep)
    s_r = np.full(n, -1, np.int32); e_r = s_r.copy(); t_r = s_r.copy()
    s_r[idx] = pos["start"]; e_r[idx] = pos["stop"]; t_r[idx] = pos["tlen"]
    keep, lo, hi = O.trim_bounds(off, rep, s_r, e_r, t_r, mode=0)
    if want_pos:
        return dict(rep=rep, strand=strand, keep=keep, lo=lo, hi=hi, rows=rows, nrep=nrep, pos=pos, first=idx), st
    return int(keep.sum()), st


def profile_paths(cfg):
    return [os.path.join(synth.HMM_DIR, f) for f in cfg["search_files"]]


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import oracle as O
    O.lib()
    import synth_big
    if args.config in synth_big.BIG_CONFIGS:
        sc = args.scale * min(1.0, 12_000 / synth_big.config(args.config, args.scale)["n_reads"])
        S1 = synth_big.BigSample(args.config, scale=sc, device="cpu")
        a, _, c = S1.block(0, S1.N, want_qual=False)
        s, o, cfg = a.numpy(), c.numpy(), synth_big.config(args.config, args.scale)
        desc = ("the same generator at %d reads / %d uniques (scale %.3g of the workload); reads/s of the whole workload is "
                "taken to be this sample's" % (S1.N, S1.U, sc))
    else:
        seq, off, which, cfg = synth.make_config(args.config, scale=args.scale)
        s, o, desc = cpu_sample(seq, off, which)
    db = O.ProfileDB(profile_paths(cfg), [cfg["left_prefix"], cfg["right_prefix"]])
    side = np.array([0 if n.startswith(cfg["left_prefix"]) else 1 for n in db.names], np.int8)
    cores = os.cpu_count()       # explicit: torchrun exports OMP_NUM_THREADS=1
    for _ in range(args.warmup):
        oracle_pipeline(O, db, side, s, o, threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_pipeline(O, db, side, s, o, threads=cores)
    dt = (time.perf_counter() - t0) / args.steps
    v = (len(o) - 1) / dt
    line = {"impl": "reference", "metric": "reads/s", "value": v, "unit": "reads/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong" if args.gpus > 1 and not args.replicas else "weak", "vs_baseline": None,
            "dtype": "u8+f32", "data": "synthetic", "config": workload_config(cfg, args, args.gpus),
            "cpu_baseline": {"value": v, "unit": "reads/s", "cores": cores, "kind": "port", "sample": desc},
            "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU oracle (oracle/liboracle.so, -O3 -fopenmp, %d host threads): a port of the reference's "
                    "vsearch + hmmsearch + ItsPosition + trim path -- neither tool is in this image; one process on the "
                    "box's host cores whatever --gpus says" % cores}
    emit(line)


def workload_config(cfg, args, world):
    length = cfg["length"]
    lmean = sum(length) / 2 if isinstance(length, tuple) else length
    if world > 1 and not args.replicas:
        par = ("ONE sample sharded over %d GPUs: block-partitioned reads, local exact derep, all-to-all of local uniques "
               "to owner key64 %% G (NCCL), owner derep + HMM search (profiles replicated), domZ all-reduce, answers "
               "through the inverse all-to-all, local trim + re-expansion" % world)
    elif world > 1:
        par = "replicas: one independent sample per GPU, no data-path collective"
    else:
        par = "one sample on one GPU"
    law = {"exact_twice": "singletons + uniques seen exactly twice", "zipf": "Zipf s=1"}.get(cfg.get("law"), "Zipf s=1")
    return {"workload": "%s: %d reads of %s bp, %d unique (%s), --region %s, profiles = %s %s_/%s_ "
                        "(F.hmm missing from the reference mount)" %
                        (WORKLOAD_NAMES.get(args.config, args.config), cfg["n_reads"], length, cfg["n_unique"], law,
                         cfg["region"], "+".join(cfg["search_files"]) if len(cfg["search_files"]) < 4 else
                         "%d taxon files" % len(cfg["search_files"]), cfg["left_prefix"][0], cfg["right_prefix"][0]),
            "taxa": cfg["taxa"], "region": cfg["region"], "scale": args.scale,
            "l2_policy": "inputs (%.0f MB of bases + qualities per step) are larger than the 126 MB L2" %
                         (2 * cfg["n_reads"] * lmean / 1e6),
            "parallelism": par}


def emit(line):
    """The ONE JSON line goes to the process's real stdout; everything else that libraries print (NCCL's version
    banner, torch warnings) was moved to stderr by main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1

DUMP_MAX_ELEMS = 1 << 20     # two legs x (2 float64 arrays of <= 8 MB + 2 float32 arrays of <= 4 MB): <= 48 MB in all


def dump_outputs(dirname, arrays):
    """Write every array as DIR/<name>.npy so that two builds can be compared output for output: bytes as float32,
    wider integers as float64 (both exact).  An array longer than DUMP_MAX_ELEMS is cut to the elements at a fixed,
    seeded, sorted sample of its indices; arrays of equal length are sampled at the same positions."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.size > DUMP_MAX_ELEMS:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a.astype(np.float32 if a.dtype.itemsize == 1 else np.float64))


def search_stages(ss_sum, sec, dsec, ds, nreads, L, pk, world=1):
    """Per-stage rates from the search / derep counters (cells summed over ranks, seconds = max over ranks)."""
    st = {
        "msv": {"ms": sec["ms_msv"] * 1e3, "gcups": ss_sum["msv_cells"] / max(sec["ms_msv"], 1e-9) / 1e9,
                "peak_gcups": pk["int_gcups"] * world, "bound": "int-alu (s16x2 DPX)"},
        "fwd_bwd_decode": {"ms": sec["ms_fwd"] * 1e3,
                           "gcups": (ss_sum["fwd_cells"] + ss_sum["bck_cells"]) / max(sec["ms_fwd"], 1e-9) / 1e9,
                           "peak_gcups": pk["fp_gcups"] * world, "bound": "fp32 fma"},
        "envelope": {"ms": sec["ms_env"] * 1e3, "gcups": ss_sum["env_cells"] / max(sec["ms_env"], 1e-9) / 1e9,
                     "peak_gcups": pk["env_gcups"] * world, "bound": "fp32 fma (+ TMA-staged scratch rows)"},
        "bias": {"ms": sec["ms_bias"] * 1e3, "rows_per_s": ss_sum["bias_rows"] / max(sec["ms_bias"], 1e-9)},
        "multidomain": {"ms": sec["ms_mdom"] * 1e3, "regions": int(ss_sum["n_multidomain_regions"]),
                        "traces_per_s": ss_sum["n_multidomain_regions"] * 200 / max(sec["ms_mdom"], 1e-9),
                        "bound": "latency / issue (200 stochastic tracebacks per flagged region, p7_domaindef)"},
        "search_total_ms": sec["ms_total"] * 1e3,
        "survival": {"pairs": int(ss_sum["n_pairs"]), "past_msv": int(ss_sum["n_past_msv"]),
                     "past_bias": int(ss_sum["n_past_bias"]), "past_fwd": int(ss_sum["n_past_fwd"]),
                     "hits": int(ss_sum["n_hits_reported"]), "domains": int(ss_sum["n_domains"]),
                     "multidomain_regions": int(ss_sum["n_multidomain_regions"])},
    }
    if dsec is not None:
        st.update({
            "derep_pack": {"ms": dsec["ms_pack"] * 1e3,
                           "gbs": ds.bytes_ascii * (1 + 0.25 + 0.125) / max(dsec["ms_pack"], 1e-9) / 1e9,
                           "peak_gbs": pk["hbm_gbs"], "bound": "hbm"},
            "derep_hash": {"ms": dsec["ms_hash"] * 1e3,
                           "gbs": (ds.bytes_ascii * 0.25 + 25.0 * nreads) / max(dsec["ms_hash"], 1e-9) / 1e9,
                           "peak_gbs": pk["hbm_gbs"], "bound": "hbm"},
            "derep_insert_verify": {"ms": (dsec["ms_insert"] + dsec["ms_verify"]) * 1e3,
                                    "gbs": nreads * (L / 2 + 28.0) / max(dsec["ms_insert"] + dsec["ms_verify"], 1e-9) / 1e9,
                                    "peak_gbs": pk["hbm_gbs"], "bound": "hbm + atomics"},
            "derep_total_ms": dsec["ms_total"] * 1e3})
    return st


def roofline_of(stages):
    dom = max(("msv", "fwd_bwd_decode", "envelope"), key=lambda k: stages[k]["ms"])
    kname = {"msv": "msv_kernel", "fwd_bwd_decode": "fb_kernel", "envelope": "env_kernel"}[dom]
    traffic, tnote = kernel_traffic(kname)
    return {"kernel": kname, "bound": "alu", "achieved": stages[dom]["gcups"], "peak": stages[dom]["peak_gcups"],
            "unit": "GCUPS", "frac": stages[dom]["gcups"] / stages[dom]["peak_gcups"], "traffic": traffic,
            "traffic_note": tnote,
            "note": "DP recurrence: fp32 / s16x2 issue-bound, not HBM or tensor; peak = MEASURED issue rate "
                    "(tools/ubench/ffma2.cu: %.3f FFMA, %.3f VIADDMNMX.S16x2 warp-instr/clk/SM) x 148 SMs x "
                    "clocks.max.sm / instructions per cell (x GPUs); HBM peak for the streaming kernels in `stages` is "
                    "MEASURED_PEAKS.json when present" % (MEASURED_FFMA_PER_CLK_SM, MEASURED_S16X2_PER_CLK_SM)}


def trim_stage(ms_bounds, ms_gather, nreads, in_bytes, out_bytes, pk):
    """SURVEY 8d K13: per read 2 L in (bases + qualities), 2 (stop - start) out, 12 B position lookup."""
    alg = 2.0 * in_bytes + 2.0 * out_bytes + 12.0 * nreads
    moved = 4.0 * out_bytes + 29.0 * nreads        # what the kernels have to touch: slices in + out, index arrays
    s = max(ms_bounds + ms_gather, 1e-9) / 1e3
    return {"ms": (ms_bounds + ms_gather), "ms_bounds": ms_bounds, "ms_gather": ms_gather,
            "gbs": alg / s / 1e9, "gbs_moved": moved / s / 1e9, "peak_gbs": pk["hbm_gbs"],
            "frac": alg / s / 1e9 / pk["hbm_gbs"], "bound": "hbm",
            "bytes_note": "gbs = SURVEY 8d's algorithmic bytes (2 L + 2 (stop-start) + 12 per read); gbs_moved counts only "
                          "the kept slices in and out plus the per-read index arrays"}


def cpu_baseline_leg(cfg, small_sample):
    from oracle import oracle as O
    s, o, desc = small_sample()
    db = O.ProfileDB(profile_paths(cfg), [cfg["left_prefix"], cfg["right_prefix"]])
    side = np.array([0 if n.startswith(cfg["left_prefix"]) else 1 for n in db.names], np.int8)
    t0 = time.perf_counter()
    oracle_pipeline(O, db, side, s, o, threads=os.cpu_count())
    dt = time.perf_counter() - t0
    return {"value": (len(o) - 1) / dt, "unit": "reads/s", "cores": os.cpu_count(), "kind": "port",
            "sample": desc, "seconds": dt}


def cli_file_to_file(seq, qual, off, cfg):
    """The real end to end a user sees: `itsxpress --fastq in.fastq --single_end --outfile out.fastq[.gz]` on this
    sample written to disk (FASTQ text in -> parse -> GPU path -> format -> [gzip] -> file out), second of two runs (page
    cache and context warm).  Host-bound; reported beside the buffer-to-buffer e2e, not instead of it."""
    import shutil
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from cli_e2e import write_fastq
    from itsxpress_b200 import main as cli
    tmp = tempfile.mkdtemp(prefix="itsx_bench_cli_")
    out = {}
    try:
        fq_in = os.path.join(tmp, "in.fastq")
        write_fastq(fq_in, seq, off, qual)
        n = len(off) - 1
        taxa = "All" if cfg["taxa"] == "All" else "Metazoa"
        for tag, name in (("plain", "out.fastq"), ("gz", "out.fastq.gz")):
            argv = ["--fastq", fq_in, "--single_end", "--outfile", os.path.join(tmp, name), "--region", cfg["region"],
                    "--taxa", taxa, "--log", os.path.join(tmp, "log.txt"), "--tempdir", tmp]
            dt = None
            for _ in range(2):
                t0 = time.perf_counter()
                cli.main(args=cli.myparser().parse_args(argv))
                dt = time.perf_counter() - t0
            out[tag] = {"reads_per_s": n / dt, "seconds": dt, "input_bytes": os.path.getsize(fq_in),
                        "output_bytes": os.path.getsize(os.path.join(tmp, name))}
        # the reference's everyday case: a single-member .fastq.gz in (one deflate stream, as a sequencer writes it), .gz out
        from cli_e2e import gzip_one_member
        gz_in = os.path.join(tmp, "in1.fastq.gz")
        with open(fq_in, "rb") as f, open(gz_in, "wb") as g:
            g.write(gzip_one_member(f.read()))
        argv = ["--fastq", gz_in, "--single_end", "--outfile", os.path.join(tmp, "out2.fastq.gz"), "--region", cfg["region"],
                "--taxa", taxa, "--log", os.path.join(tmp, "log.txt"), "--tempdir", tmp]
        for _ in range(2):
            t0 = time.perf_counter()
            cli.main(args=cli.myparser().parse_args(argv))
            dt = time.perf_counter() - t0
        out["gz_in_gz_out"] = {"reads_per_s": n / dt, "seconds": dt, "input_bytes": os.path.getsize(gz_in),
                               "output_bytes": os.path.getsize(os.path.join(tmp, "out2.fastq.gz")),
                               "host_cores": os.cpu_count()}
        out["note"] = ("wall clock of itsxpress_b200.main.main(); bound by FASTQ parsing / formatting on the host; .gz output is "
                       "compressed on the GPU (itsx_gzip_compress); a .gz input is ONE deflate stream inflated on all host "
                       "cores (csrc/inflate_host.cpp)")
    except BaseException as e:          # the CLI ends in SystemExit on failure; the bench line must still come out
        out["error"] = "%s: %s" % (type(e).__name__, e)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return out


# ---------------------------------------------------------------------------------------------------------------
def run_single(args, rank, world, local):
    """One sample per GPU (N = 1, or --replicas)."""
    import torch
    import torch.distributed as dist
    from itsxpress_b200 import _lib
    ctx = _lib.Context(local)
    import synth_big
    if args.config in synth_big.BIG_CONFIGS:
        S = synth_big.BigSample(args.config, scale=args.scale, device="cuda:%d" % local)
        cfg = S.cfg
        a, b, c_ = S.block(0, S.N)
        seq, qual, off, which = a.cpu().numpy(), b.cpu().numpy(), c_.cpu().numpy(), None
        del a, b, c_, S
        torch.cuda.empty_cache()
    else:
        seq, off, which, cfg = synth.make_config(args.config, seed=2 * 1_000_003 + rank, scale=args.scale)
        qual = synth.make_quals(77 + rank, off)
    nreads = len(off) - 1
    ctx.load_profiles(profile_paths(cfg), [cfg["left_prefix"], cfg["right_prefix"]])
    ctx.set_sides_by_prefix(cfg["left_prefix"], cfg["right_prefix"])
    prm = _lib.default_params()

    # pinned host staging for the e2e leg: bases, qualities, offsets in; kept index, offsets, bases, qualities out
    tot = int(off[-1])
    a64 = lambda x: (x + 63) // 64 * 64
    pin_in = _lib.PinnedBuffer(2 * a64(tot) + off.nbytes + 64)
    pseq = pin_in.array(np.uint8, tot)
    pqual = pin_in.array(np.uint8, tot, offset=a64(tot))
    poff = pin_in.array(np.int64, off.size, offset=2 * a64(tot))
    pseq[:] = seq
    pqual[:] = qual
    poff[:] = off
    pin_out = _lib.PinnedBuffer(2 * a64(tot) + a64(nreads * 4) + (nreads + 1) * 8 + 64)
    outs = dict(rep=None, out_seq=pin_out.array(np.uint8, tot), out_qual=pin_out.array(np.uint8, tot, offset=a64(tot)),
                kept_index=pin_out.array(np.int32, nreads, offset=2 * a64(tot)),
                out_off=pin_out.array(np.int64, nreads + 1, offset=2 * a64(tot) + a64(nreads * 4)))

    ext = torch.cuda.ExternalStream(ctx.stream, device=local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ext):
            e0.record()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        with torch.cuda.stream(ext):
            e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        barrier()
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    # ---- resident leg (value): bases + qualities + offsets already in HBM ----
    ctx.reads_upload(pseq, poff)
    ctx.quals_upload(pqual)
    skeys = ("ms_msv", "ms_bias", "ms_fwd", "ms_mdom", "ms_env", "ms_final", "ms_total")
    dkeys = ("ms_pack", "ms_hash", "ms_insert", "ms_verify", "ms_compact", "ms_total")
    stage = {k: 0.0 for k in skeys}
    dstage = {k: 0.0 for k in dkeys}
    tstage = {"ms_trim": 0.0, "ms_gather": 0.0}
    last = {}

    def step_resident():
        st = ctx.run_resident(prm)
        ss, ds = ctx.search_stats(), ctx.derep_stats()
        for k in stage:
            stage[k] += getattr(ss, k)
        for k in dstage:
            dstage[k] += getattr(ds, k)
        for k in tstage:
            tstage[k] += getattr(st, k)
        last["run"], last["search"], last["derep"] = st, ss, ds

    for _ in range(max(args.warmup, 3)):
        step_resident()
    for d in (stage, dstage, tstage):
        for k in d:
            d[k] = 0.0
    clk = ClockSampler(local)
    clk.start()
    l0 = ctx.launch_count()
    ms_dev, ms_wall = timed(step_resident, args.steps)
    launches = ctx.launch_count() - l0
    # what the last resident step left on the device (untimed; the e2e leg below overwrites it)
    resident_out = None
    if rank == 0 and args.dump_outputs:
        resident_out = dict(zip(("kept_index", "out_off", "out_seq", "out_qual"), ctx.run_fetch()))
    # ---- e2e leg: host buffers in, trimmed records out ----
    rs_e2e = None
    for _ in range(2):
        ctx.run_trim(pseq, pqual, poff, prm, out=outs)

    def step_e2e():
        last["e2e_out"], last["e2e"] = ctx.run_trim(pseq, pqual, poff, prm, out=outs)

    ms_e2e_dev, ms_e2e_wall = timed(step_e2e, args.steps)
    clocks = clk.stop()
    rs_e2e = last["e2e"]
    if rank == 0 and args.dump_outputs:
        arrays = {}
        for leg, out, st in (("resident", resident_out, last["run"]), ("e2e", last["e2e_out"], rs_e2e)):
            arrays.update({"%s_%s" % (leg, k): out[k] for k in ("kept_index", "out_off", "out_seq", "out_qual")})
            arrays["%s_counts" % leg] = np.array([st.n_reads, st.n_unique, st.n_kept, st.out_bytes], np.int64)
        dump_outputs(args.dump_outputs, arrays)

    total_reads = nreads * world
    value = total_reads / (ms_dev / 1e3 / args.steps)
    e2e_v = total_reads / (max(ms_e2e_dev, ms_e2e_wall) / 1e3 / args.steps)
    ss, ds, rs = last["search"], last["derep"], last["run"]
    pk = peaks()
    K = args.steps
    sec = {k: v / 1e3 / K for k, v in stage.items()}
    dsec = {k: v / 1e3 / K for k, v in dstage.items()}
    L = sum(cfg["length"]) / 2 if isinstance(cfg["length"], tuple) else cfg["length"]
    stages = search_stages(ss.asdict(), sec, dsec, ds, nreads, L, pk)
    stages["trim_gather"] = trim_stage(tstage["ms_trim"] / K, tstage["ms_gather"] / K, nreads, tot, int(rs.out_bytes), pk)
    roof = roofline_of(stages)

    cli_extra = None
    if rank == 0 and world == 1 and not args.no_cli and nreads <= 2_000_000:
        cli_extra = cli_file_to_file(seq, qual, off, cfg)
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        if which is not None:
            cpu = cpu_baseline_leg(cfg, lambda: cpu_sample(seq, off, which))
        else:
            k = min(nreads, 12_000)
            cpu = cpu_baseline_leg(cfg, lambda: (seq[:off[k]].copy(), off[:k + 1].copy(),
                                                 "the first %d reads of the workload; reads/s of the whole workload is taken "
                                                 "to be this sample's" % k))

    if rank == 0:
        h2d = int(2 * tot + off.nbytes)
        d2h = int(2 * rs_e2e.out_bytes + rs_e2e.n_kept * 4 + (rs_e2e.n_kept + 1) * 8)
        line = {"metric": "reads/s", "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8/s16x2 (MSV) + f32 (Forward/Backward)",
                "data": "synthetic", "config": workload_config(cfg, args, world), "clocks": clocks,
                "e2e": {"value": e2e_v, "unit": "reads/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": max(ms_e2e_dev, ms_e2e_wall) / args.steps,
                        "call": "itsx_run_trim: bases + qualities + offsets up, trimmed bases + qualities + offsets + "
                                "kept index down (pinned host buffers)",
                        "ms_h2d": rs_e2e.ms_h2d, "ms_d2h": rs_e2e.ms_d2h},
                "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu, "stages": stages,
                "hmm_gcups": {"msv": stages["msv"]["gcups"], "fwd_bwd": stages["fwd_bwd_decode"]["gcups"],
                              "envelope": stages["envelope"]["gcups"]},
                "result": {"n_unique": int(rs.n_unique), "n_kept": int(rs.n_kept), "out_bytes": int(rs.out_bytes),
                           # checksums of what the last e2e step returned (equal across builds of the same path)
                           "crc32": {k: zlib.crc32(last["e2e_out"][k].tobytes())
                                     for k in ("kept_index", "out_off", "out_seq", "out_qual")},
                           "n_selected_multidomain": int(ss.n_selected_multidomain)},
                "extra": {"cli_file_to_file": cli_extra}}
        emit(line)


_KEEP = []      # pinned allocations stay alive for the life of the process (numpy views do not own them)


def pinned_or_pageable(_lib, nbytes):
    """Page-locked staging up to 4 GB per buffer; beyond that (configs[3]: 10 GB per rank and direction) plain host memory --
    eight ranks pinning 150 GB of one host is not what a user's reader would do either, and the copies are < 5 % of those
    steps."""
    try:
        if nbytes > (4 << 30):
            raise MemoryError
        _KEEP.append(_lib.PinnedBuffer(nbytes))
        return _KEEP[-1]
    except MemoryError:
        class _Pageable:
            def __init__(self, n):
                self.buf = np.empty(n, np.uint8)

            def array(self, dtype=np.uint8, count=None, offset=0):
                dtype = np.dtype(dtype)
                return self.buf[offset:offset + count * dtype.itemsize].view(dtype)
        return _Pageable(nbytes)


def load_block(args, rank, world, local, _lib, block_range):
    """This rank's block of the workload in pinned host memory: (bseq, bqual, boff, lo, hi, n, total_bytes, cfg, full)
    where full() returns the whole sample (seq, qual, off, which) when it is small enough to check against one GPU."""
    a64 = lambda x: (x + 63) // 64 * 64
    import synth_big
    if args.config in synth_big.BIG_CONFIGS:
        import torch
        S = synth_big.BigSample(args.config, scale=args.scale, device="cuda:%d" % local)
        cfg, n = S.cfg, S.N
        lo, hi = block_range(n, rank, world)
        seq_d, qual_d, off_d = S.block(lo, hi)
        tb, nb = int(off_d[-1].item()), hi - lo
        pin = pinned_or_pageable(_lib, 2 * a64(tb) + (nb + 1) * 8 + 64)
        bseq, bqual = pin.array(np.uint8, tb), pin.array(np.uint8, tb, offset=a64(tb))
        boff = pin.array(np.int64, nb + 1, offset=2 * a64(tb))
        torch.from_numpy(bseq).copy_(seq_d)
        torch.from_numpy(bqual).copy_(qual_d)
        torch.from_numpy(boff).copy_(off_d)
        tot = torch.tensor([float(tb)], dtype=torch.float64, device="cuda")
        if world > 1:
            torch.distributed.all_reduce(tot)
        del seq_d, qual_d, off_d
        torch.cuda.empty_cache()

        def full():
            if n > 4_000_000:
                return None
            S0 = synth_big.BigSample(args.config, scale=args.scale, device="cuda:%d" % local)
            a, b, c = S0.block(0, n)
            r = (a.cpu().numpy(), b.cpu().numpy(), c.cpu().numpy(), None)
            del a, b, c, S0
            torch.cuda.empty_cache()
            return r

        def small():
            """the same generator at a size the CPU oracle finishes in ~10-20 s"""
            sc = args.scale * min(1.0, 12_000 / n)
            S1 = synth_big.BigSample(args.config, scale=sc, device="cpu")
            a, _, c = S1.block(0, S1.N, want_qual=False)
            return a.numpy(), c.numpy(), ("the same generator at %d reads / %d uniques (scale %.3g of the workload); reads/s "
                                          "of the whole workload is taken to be this sample's" % (S1.N, S1.U, sc))
        return bseq, bqual, boff, lo, hi, n, int(tot.item()), cfg, full, small
    seq, off, which, cfg = synth.make_config(args.config, scale=args.scale)
    qual = synth.make_quals(77, off)
    n = len(off) - 1
    lo, hi = block_range(n, rank, world)
    b0, b1 = int(off[lo]), int(off[hi])
    nb, tb = hi - lo, b1 - b0
    pin = pinned_or_pageable(_lib, 2 * a64(tb) + (nb + 1) * 8 + 64)
    bseq, bqual = pin.array(np.uint8, tb), pin.array(np.uint8, tb, offset=a64(tb))
    boff = pin.array(np.int64, nb + 1, offset=2 * a64(tb))
    bseq[:] = seq[b0:b1]
    bqual[:] = qual[b0:b1]
    boff[:] = off[lo:hi + 1] - b0

    def small():
        s_, o_, desc = cpu_sample(seq, off, which)
        return s_, o_, desc
    return bseq, bqual, boff, lo, hi, n, int(off[-1]), cfg, (lambda: (seq, qual, off, which)), small


# ---------------------------------------------------------------------------------------------------------------
def run_sharded_bench(args, rank, world, local):
    """ONE sample, block-partitioned over the ranks (itsxpress_b200.distributed.run_sharded on libitsx_b200).
    value: the rank's block resident in HBM; e2e: the block in pinned host memory, trimmed records back to the host.
    Time = max over ranks (CUDA events on torch's stream around host-synchronous phases, and the wall clock)."""
    import torch
    import torch.distributed as dist
    from itsxpress_b200 import _lib
    from itsxpress_b200.distributed import PHASES, Comm, GpuEngine, block_range, run_sharded
    bseq, bqual, boff, lo, hi, n, total_bytes, cfg, full_sample, small_sample = load_block(args, rank, world, local, _lib,
                                                                                         block_range)
    nb, tb = hi - lo, int(boff[-1])
    paths, pre = profile_paths(cfg), [cfg["left_prefix"], cfg["right_prefix"]]
    local_ctx, owner_ctx = _lib.Context(local), _lib.Context(local)
    owner_ctx.load_profiles(paths, pre)
    owner_ctx.set_sides_by_prefix(*pre)
    prm = _lib.default_params()
    prm.domz_upper = n               # any profile's domZ <= the sample's read count (compact row mode, see itsx_b200.h)
    comm = Comm()
    eng = GpuEngine(local_ctx, owner_ctx, prm)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    skeys = ("ms_msv", "ms_bias", "ms_fwd", "ms_mdom", "ms_env", "ms_final", "ms_total")
    last = {}

    def timed(fn, steps, phases, stage):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        for _ in range(steps):
            last["out"] = fn(phases)
            if stage is not None:
                ss = owner_ctx.search_stats()
                for k in skeys:
                    stage[k] += getattr(ss, k)
                last["search"] = ss
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        barrier()
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    # pinned worst-case outputs of the e2e leg (every read kept whole)
    a64 = lambda x: (x + 63) // 64 * 64
    pout = pinned_or_pageable(_lib, 2 * a64(tb) + a64(nb * 4) + (nb + 1) * 8 + 64)
    gout = dict(out_seq=pout.array(np.uint8, tb), out_qual=pout.array(np.uint8, tb, offset=a64(tb)),
                kept_index=pout.array(np.int32, nb, offset=2 * a64(tb)),
                out_off=pout.array(np.int64, nb + 1, offset=2 * a64(tb) + a64(nb * 4)))
    # ---- value: block resident, results left in HBM ----
    eng.upload(bseq, boff, bqual)
    step_res = lambda ph: run_sharded(eng, comm, None, None, lo, phases=ph, want_rep=False, gather="device")
    for _ in range(max(args.warmup, 3)):
        step_res(None)
    clk = ClockSampler(local)
    clk.start()
    l0 = local_ctx.launch_count() + owner_ctx.launch_count()
    phases, stage = {}, {k: 0.0 for k in skeys}
    comm.bytes_sent = {}
    ms_dev, ms_wall = timed(step_res, args.steps, phases, stage)
    launches = local_ctx.launch_count() + owner_ctx.launch_count() - l0
    sent = dict(comm.bytes_sent)
    out_res = last["out"]
    # ---- e2e: host buffers in (H2D inside), trimmed records out (D2H inside) ----
    eng.resident = eng.resident_qual = False
    step_e2e = lambda ph: run_sharded(eng, comm, bseq, boff, lo, phases=ph, want_rep=False, gather=True, qual=bqual,
                                      gather_out=gout)
    for _ in range(2 if n <= 20_000_000 else 1):     # (kernels and allocations are warm from the resident leg)
        step_e2e(None)
    ph_e2e = {}
    ms_e2e_dev, ms_e2e_wall = timed(step_e2e, args.steps, ph_e2e, None)
    clocks = clk.stop()
    out = last["out"]
    K = args.steps

    # ---- reductions over ranks ----
    ss = last["search"].asdict()
    sum_keys = ("n_seq", "n_pairs", "n_past_msv", "n_past_bias", "n_past_fwd", "n_hits_reported", "n_domains",
                "n_multidomain_regions", "msv_cells", "bias_rows", "fwd_cells", "bck_cells", "env_cells")
    vsum = torch.tensor([float(ss[k]) for k in sum_keys] +
                        [float(len(out["kept_index"])), float(len(out["out_seq"])), float(launches),
                         float((out["kept_index"].astype(np.int64) + lo).sum()),
                         float(out["n_local_unique"]), float(tb)], dtype=torch.float64, device="cuda")
    dist.all_reduce(vsum, op=dist.ReduceOp.SUM)
    vmax = torch.tensor([stage[k] for k in skeys] + [phases.get(p, 0.0) for p in PHASES] +
                        [ph_e2e.get(p, 0.0) for p in PHASES] + [float(out["n_owned"]), float(tb)],
                        dtype=torch.float64, device="cuda")
    vmin = -vmax.clone()
    dist.all_reduce(vmax, op=dist.ReduceOp.MAX)
    dist.all_reduce(vmin, op=dist.ReduceOp.MAX)
    vmin = -vmin
    sent_t = torch.tensor([float(sent.get(k, 0)) for k in ("records", "bases", "answers")], dtype=torch.float64,
                          device="cuda")
    dist.all_reduce(sent_t, op=dist.ReduceOp.MAX)
    crc = torch.tensor([zlib.crc32(out["out_seq"].tobytes()), zlib.crc32(out["out_qual"].tobytes())], dtype=torch.int64,
                       device="cuda")
    crcs = [torch.zeros_like(crc) for _ in range(world)]
    dist.all_gather(crcs, crc)

    if rank == 0:
        vs, vm, vn = vsum.tolist(), vmax.tolist(), vmin.tolist()
        ss_sum = dict(zip(sum_keys, vs[:len(sum_keys)]))
        n_kept, out_bytes, launches_all, kept_cksum, nu_local_sum, _ = vs[len(sum_keys):]
        sec = {k: vm[i] / 1e3 / K for i, k in enumerate(skeys)}
        ph = {p: vm[len(skeys) + i] / K * 1e3 for i, p in enumerate(PHASES)}
        ph2 = {p: vm[len(skeys) + len(PHASES) + i] / K * 1e3 for i, p in enumerate(PHASES)}
        own_max, tb_max = vm[-2], vm[-1]
        own_min, tb_min = vn[-2], vn[-1]
        pk = peaks()
        L = sum(cfg["length"]) / 2 if isinstance(cfg["length"], tuple) else cfg["length"]
        stages = search_stages(ss_sum, sec, None, None, n, L, pk, world)
        roof = roofline_of(stages)
        # ---- the same sample on ONE GPU (untimed): identical kept reads, identical trimmed bytes ----
        whole = full_sample()
        equal, check = None, "skipped: the sample is too large for one untimed one-GPU pass inside the bench"
        if whole is not None:
            seq, qual, off, _ = whole
            single, st1 = owner_ctx.run_trim(seq, qual, off, prm)
            ki1, oo1 = single["kept_index"], single["out_off"]
            ok = int(st1.n_kept) == int(n_kept) and int(st1.out_bytes) == int(out_bytes) and \
                int(st1.n_unique) == int(out["n_unique_global"]) and int(ki1.astype(np.int64).sum()) == int(kept_cksum)
            for r in range(world):
                rlo, rhi = block_range(n, r, world)
                a, b = np.searchsorted(ki1, rlo), np.searchsorted(ki1, rhi)
                want = (zlib.crc32(single["out_seq"][oo1[a]:oo1[b]].tobytes()),
                        zlib.crc32(single["out_qual"][oo1[a]:oo1[b]].tobytes()))
                ok = ok and tuple(int(x) for x in crcs[r].tolist()) == want
            if not ok:
                raise SystemExit("bench.py: the sharded result differs from the one-GPU result on the same sample "
                                 "(n_kept %d vs %d, n_unique %d vs %d)" % (n_kept, st1.n_kept, out["n_unique_global"],
                                                                          st1.n_unique))
            equal = True
            check = ("n_unique, n_kept, trimmed byte count, kept-index checksum and per-block CRC32 of the trimmed bases and "
                     "qualities equal itsx_run_trim on one GPU (rank 0, untimed)")
        ex_s = max(ph["exchange"], 1e-6) / 1e3
        an_s = max(ph["answers_exchange"], 1e-6) / 1e3
        value = n / (max(ms_dev, ms_wall) / 1e3 / K)
        e2e_v = n / (max(ms_e2e_dev, ms_e2e_wall) / 1e3 / K)
        cpu = None if args.no_cpu_baseline else cpu_baseline_leg(cfg, small_sample)
        search_ms = ph["search_stage1"] + ph["search_stage2"]
        line = {"metric": "reads/s", "value": value, "unit": "reads/s", "n_gpus": world, "steps": K,
                "warmup": max(args.warmup, 3), "ms_per_step": max(ms_dev, ms_wall) / K, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "u8/s16x2 (MSV) + f32 (Forward/Backward)",
                "data": "synthetic", "config": workload_config(cfg, args, world), "clocks": clocks,
                "e2e": {"value": e2e_v, "unit": "reads/s", "h2d_bytes_per_step": int(2 * total_bytes + (n + world) * 8),
                        "d2h_bytes_per_step": int(2 * out_bytes + n_kept * 4 + (n_kept + world) * 8),
                        "ms_per_step": max(ms_e2e_dev, ms_e2e_wall) / K,
                        "call": "run_sharded(GpuEngine): every rank's block goes up from pinned host memory, its "
                                "trimmed bases + qualities + offsets + kept index come back",
                        "phases_ms": ph2},
                "gpu_launches": int(launches_all), "roofline": roof, "cpu_baseline": cpu, "stages": stages,
                "phases_ms": dict(ph, note="max over ranks, mean over the timed steps; host-synchronous phases of "
                                           "itsxpress_b200.distributed.run_sharded, block resident in HBM"),
                "limiting_phase": max(ph, key=ph.get),
                "collectives": {
                    "forward_all_to_all": {"bytes_per_rank_max": int((sent_t[0] + sent_t[1]) / K),
                                           "records_bytes": int(sent_t[0] / K), "bases_bytes": int(sent_t[1] / K),
                                           "ms": ph["exchange"],
                                           "gbs_per_rank": (sent_t[0].item() + sent_t[1].item()) / K / ex_s / 1e9,
                                           "nvlink_peak_gbs": NVLINK_GBS,
                                           "note": "2 G split sizes, then records (8 B / local unique) and bases; "
                                                   "latency-bound at this size"},
                    "domz_all_reduce": {"bytes": 8 * (int(ss["n_prof"]) + 1), "ms": ph["domz_allreduce"]},
                    "answers_all_to_all": {"bytes_per_rank_max": int(sent_t[2] / K), "ms": ph["answers_exchange"],
                                           "gbs_per_rank": sent_t[2].item() / K / an_s / 1e9, "nvlink_peak_gbs": NVLINK_GBS}},
                "balance": {"classes_per_owner_max": int(own_max), "classes_per_owner_min": int(own_min),
                            "block_bytes_max": int(tb_max), "block_bytes_min": int(tb_min),
                            "local_uniques_sum": int(nu_local_sum),
                            "note": "owner = key64 % G: classes (and their bases, reads here have one length) spread "
                                    "within max/min above; search time follows classes per owner"},
                "hmm_gcups": {"msv": stages["msv"]["gcups"], "fwd_bwd": stages["fwd_bwd_decode"]["gcups"],
                              "envelope": stages["envelope"]["gcups"]},
                "search_share": search_ms / max(sum(ph[p] for p in PHASES), 1e-9),
                "result": {"n_unique": int(out["n_unique_global"]), "n_kept": int(n_kept), "out_bytes": int(out_bytes),
                           "equals_single_gpu": equal, "check": check}}
        emit(line)
    barrier()


def main():
    global _REAL_STDOUT
    import faulthandler
    faulthandler.enable()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (testing only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cli", action="store_true", help="skip the file-to-file command-line timing (extra.cli_file_to_file)")
    import synth_big
    ap.add_argument("--config", default="c2", choices=sorted(set(synth.CONFIGS) | set(synth_big.BIG_CONFIGS)),
                    help="workload: c2 = BASELINE configs[1] (the headline); c3 / c4 = configs[2] / [3]; c4s / c3s = "
                         "scaled shapes of them")
    ap.add_argument("--replicas", action="store_true",
                    help="N > 1: one independent sample per rank (weak scaling, no collective) instead of ONE sample "
                         "sharded over the ranks")
    ap.add_argument("--sharded", action="store_true", help="accepted for compatibility: sharding is the N > 1 default")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step of each timed leg returned (kept index, "
                         "offsets, trimmed bases and qualities, counts) as DIR/<leg>_<name>.npy in float32 / float64; "
                         "arrays longer than %d elements as a fixed, seeded sample" % DUMP_MAX_ELEMS)
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or (world > 1 and not args.replicas)):
        ap.error("--dump-outputs writes the outputs of one GPU's sample: use it on the GPU path with one GPU or "
                 "--replicas")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if world > 1 and not args.replicas:
        run_sharded_bench(args, rank, world, local)
    else:
        run_single(args, rank, world, local)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
