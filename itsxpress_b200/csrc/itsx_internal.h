// itsx_internal.h -- shared declarations of libitsx_b200 (host C++ and CUDA translation units).
// Public C ABI: include/itsx_b200.h.  Nothing here is visible to callers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <algorithm>
#include <string>
#include <vector>
#include "../../include/itsx_b200.h"

#define ITSX_NCODE 16   // residue codes: 0..3 ACGT, 4..14 RYMKSWHBVDN, 15 = illegal/other
#define ITSX_KP ((ITSX_MAXM + 2) / 2)   // 23 s16x2 node pairs per MSV row
#define ITSX_NT 7
enum { T_MM = 0, T_MI, T_MD, T_IM, T_II, T_DM, T_DD, T_BM };   // T_BM: B->M_k entry, 8th column
enum { EV_MMU = 0, EV_MLAMBDA, EV_VMU, EV_VLAMBDA, EV_FTAU, EV_FLAMBDA };

// ---- one configured profile on the host (hmmfile.cpp) ---------------------------------
struct HostProfile {
    std::string name;
    int   M = 0;
    std::vector<float> mat;     // (M+1)*4 match emission probabilities (row 0 unused)
    std::vector<float> t;       // (M+1)*7 transition probabilities, row 0 = begin node
    float compo[4] = {0.25f, 0.25f, 0.25f, 0.25f};
    float ev[6] = {0, 0, 0, 0, 0, 0};
    // search profile, local multihit (SURVEY A.3)
    std::vector<float> msc;     // (M+1)*16 match log-odds, nats
    std::vector<float> e;       // (M+1)*16 match odds
    std::vector<float> bm;      // (M+2) B->M_k probability
    std::vector<float> tp;      // (M+2)*7 transition probabilities out of node k (0 for k=0, k>=M)
    // MSV byte profile (SURVEY A.4 step 1)
    std::vector<uint8_t> cost;  // (M+1)*16 biased byte costs
    int   bias_b = 0, base_b = 190, tbm_b = 0, tec_b = 0;
    float scale_b = 0.f;
    float eo[ITSX_NCODE][2];    // bias-filter emission odds [code][state]
};
int  hmmfile_append(const char *path, const char *const *prefixes, int nprefix,
                    std::vector<HostProfile> &out, std::string &err);
uint8_t msv_unbiased_byteify(float scale_b, float sc);

// ---- device-side profile tables ------------------------------------------------------------
// transitions + entry, node-major: tp[k] = {MM, MI, MD, IM, II, DM, DD, BM_k}, k = 0..MAXM+1.
// Passed BY VALUE as a __grid_constant__ kernel argument so that every FFMA reads its
// coefficient straight from the constant bank (no load instruction in the DP inner loop).
// Coefficients are additionally laid out in the order the unrolled DP loops consume them, so that every
// uniform load (LDCU.128 / .64) is fully used and no value is shared between distant cells:
//   Forward  pass 1 (M, I of row i):  fa[k] = {BM_k, MM_{k-1}, IM_{k-1}, DM_{k-1}}   fi[k] = {II_k, MI_k}
//            pass 2 (D chain):        fd[k] = {DD_{k-1}, MD_{k-1}}
//   Backward pass 1 (B sum):          bm[k] = BM_k
//            pass 2 (M, I, D):        ba[k] = {IM_k, II_k, MM_k, MI_k}               bd[k] = {DM_k, DD_k, MD_k, 0}
struct alignas(16) ProfConst {
    float fa[ITSX_MAXM + 1][4];
    float fi[ITSX_MAXM + 1][2];
    float fd[ITSX_MAXM + 1][2];
    float ba[ITSX_MAXM + 1][4];
    // node k lives at index k - 1 so that four consecutive nodes are one aligned 128-bit uniform load (LDCU.128)
    float bd0[ITSX_MAXM + 3], bd1[ITSX_MAXM + 3], bd2[ITSX_MAXM + 3];   // D->M, D->D, M->D out of node k
    float bm[ITSX_MAXM + 3];                                            // B->M_k entry
};
// per-profile scalars used by the filter kernels
struct ProfScalars {
    int32_t M, bias, base, tbm, tec, side, pad0, pad1;
    float   scale_b;
    float   ev[6];
    float   pad2;
    float   eo[ITSX_NCODE][2];
};

// one survivor of the filter cascade (worklist entry); arrays are struct-of-arrays on device
struct DomRec {
    int32_t seq, prof, ienv, jenv, tlen, dom_idx;
    float   bitscore, envsc, domcorrection, seq_score;
    double  lnP, seq_lnP;
    int32_t is_multidomain, pair_reported;
};

// one int64 of a caller buffer that may live on the host or on the device (every caller buffer of the C ABI may be
// device memory: copies use cudaMemcpyDefault)
inline int64_t itsx_peek_i64(const int64_t *p)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) == cudaSuccess && (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged)) {
        int64_t v = 0;
        cudaMemcpy(&v, p, 8, cudaMemcpyDefault);
        return v;
    }
    cudaGetLastError();
    return *p;
}

// growable device buffer (library-owned; grows geometrically, never shrinks)
struct DevBuf {
    void  *p = nullptr;
    size_t cap = 0;
    ~DevBuf();
    cudaError_t ensure(size_t bytes, bool keep = false, cudaStream_t st = 0);
    template <typename T> T *as() const { return (T *)p; }
};

struct itsx_ctx {
    int device = 0, sm_count = 0, cc_major = 0, cc_minor = 0;
    size_t mem_total = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    int64_t launches = 0;

    // profiles
    std::vector<HostProfile> prof;
    std::vector<int8_t> side;
    bool prof_dirty = true;
    DevBuf d_msvtab;      // uint32 [P][ITSX_KP][16]: (bias - cost) of nodes (2j+1, 2j+2) as s16x2
    DevBuf d_etab;        // float  [P][ITSX_MAXM+1][16]: match odds
    DevBuf d_pscal;       // ProfScalars [P]
    DevBuf d_logsum;      // float [16000] p7_FLogsum table
    DevBuf d_vtab, d_xwmove, d_vneed, d_vpass;   // Viterbi filter: int32 [P][VIT_WORDS] tables, int16 xw_move per length, per-entry flags
    DevBuf d_mdtab;       // float [P][ITSX_MAXM+2][8]: transitions out of node k + B->M_k (multidomain resolver)
    DevBuf d_mdlist, d_envdc, d_n2reg, d_mdreg, d_mdres, d_mdscratch[2], d_mdcell[2], d_mdtrace[2];   // multidomain worklist (+ count), per-envelope trace domcorrection, per-entry region n2sc sum
    std::vector<ProfConst> pconst;   // host copies handed to the per-profile launches

    // reads of the last derep (device resident)
    int64_t nreads = 0, total_bases = 0;
    DevBuf d_ascii, d_off;            // uint8 [total], int64 [nreads+1]
    DevBuf d_pack2, d_exc;            // 2-bit packed stream (uint32 / 16 bases), non-ACGT bit mask (uint32 / 32 bases)
    DevBuf d_key, d_flags;            // uint64 key per read, uint8 flags (bit0: has non-ACGT, bit1: canonical = revcomp)
    DevBuf d_table;                   // hash slots
    DevBuf d_rep, d_strand, d_abund;  // int32 rep_index, uint8 strand, int32 count at representative
    DevBuf d_collide;                 // collided read list
    DevBuf d_uid, d_first;            // int32 unique id per read; int32 first_read per unique
    DevBuf d_tmp;                     // cub temp storage
    DevBuf d_gz_in, d_gz_tok, d_gz_out, d_gz_meta, d_gz_pack;   // gzip writer (deflate.cu): text, tokens, blocks, sizes / CRCs / offsets, framed members
    DevBuf d_counters;                // uint64 [32] device counters (see CNT_* below)
    DevBuf d_lut;                     // uint8 [256] ASCII -> residue code
    int64_t n_unique = 0;
    // several samples in one pass (QIIME 2 artifacts, q2_itsxpress.py:273-333: derep, Z and domZ are per sample):
    // sample id per read; classes never span samples, reported-hit counts are per (sample, profile)
    DevBuf d_sample, d_seq_sample;     // int32 per read / per searched sequence
    int32_t n_samples = 1;
    bool have_samples = false;
    bool map_external = false;        // d_uid installed by itsx_trim_set_map (no resident read bytes)
    int key_bits = 64;
    itsx_derep_stats dstats{};
    // clustering of the derep classes (cluster.cu): while cl_active, d_uid maps reads to centroid rows and the search set is
    // the cl_ncent centroids; d_cl_class keeps the exact class of every read
    bool cl_active = false;
    int64_t cl_ncent = 0;
    int cl_key_bits = 64;
    itsx_cluster_stats clstats{};
    DevBuf d_cl_class, d_cl_order, d_cl_u, d_cl_tab, d_cl_r, d_cl_seg, d_cl_key, d_cl_val, d_cl_cnt, d_cl_cand, d_cl_acc;
    DevBuf d_cl_edge, d_cl_beg, d_cl_state, d_cl_rres, d_cl_row, d_cl_out, d_cl_crow;

    // searched sequences (uniques): nibble-coded residues
    int64_t nseq = 0;
    int     Lmax = 0;
    DevBuf d_seqw, d_seqwoff, d_seqlen;   // uint32 words (8 residues each), int64 word offset [nseq+1], int32 length
    DevBuf d_order;                       // int32: sequences of the searched shard sorted by length (+ sort scratch)
    DevBuf d_nullsc, d_tjb;               // per-length tables: float nullsc[Lmax+1], uint8 tjb[Lmax+1]
    std::vector<int32_t> h_seqlen;
    int64_t shard_first = 0, shard_n = -1;

    // search state / results
    itsx_search_params prm{};
    itsx_search_stats sstats{};
    DevBuf d_doms;                        // DomRec [ndom]
    int64_t ndom = 0;
    DevBuf d_nrep;                        // int32 [P] reported hits per profile (domZ)
    std::vector<int32_t> h_nrep;
    bool stage1_done = false, stage2_done = false;
    bool compact = false;                 // keep_rows mode 2 of the last stage 1 (see include/itsx_b200.h)
    bool stage2_applied = false;
    int64_t n_certain_rows = 0;
    DevBuf d_selmulti;                    // uint8 [2][nseq]: the selected left / right row came out of a multidomain region
    DevBuf d_pos;                         // int32 [9][nseq] start, stop, tlen, lsc, lfrom, lto, rsc, rfrom, rto
    DevBuf d_best;                        // uint64 [2][nseq]
    int64_t npos = 0;
    bool pos_valid = false;

    // scratch of the search stages
    DevBuf d_msvres, d_flag, d_scan, d_list, d_bounds, d_filtersc, d_list2, d_fsc2;
    DevBuf d_fwdsc, d_fbscale, d_spec, d_ndom, d_env, d_envoff, d_envwork, d_envout, d_envscratch, d_pairout;
    // paired-end merge (merge.cu): inputs, slotted and compacted outputs of the last itsx_merge_pairs
    DevBuf d_mg_fseq, d_mg_fqual, d_mg_foff, d_mg_rseq, d_mg_rqual, d_mg_roff, d_mg_tabs, d_mg_hist;
    DevBuf d_mg_mlen, d_mg_reason, d_mg_sseq, d_mg_squal, d_mg_flag, d_mg_len64, d_mg_kscan, d_mg_lscan;
    DevBuf d_mg_idx, d_mg_ooff, d_mg_oseq, d_mg_oqual;
    int64_t mg_npairs = 0, mg_nmerged = 0, mg_total = 0;
    bool mg_tabs_ready = false;
    itsx_merge_params mg_tabs_prm{};
    itsx_merge_stats mgstats{};

    // qualities of the resident reads (itsx_quals_upload, a streamed upload with qualities)
    DevBuf d_qual;
    bool qual_resident = false;
    // streamed upload (itsx_reads_begin / append / end): reads and bases appended so far, every chunk brought qualities
    bool stream_open = false, stream_qual = false;
    int64_t stream_reads = 0, stream_bases = 0;
    // trim (trim.cu): keep / lo / hi of the last trim_bounds_dev over r_n reads with offsets r_off, its kept count and
    // output bytes; the slices of the last trim_gather_dev (r_gathered; r_gathered_qual: qualities too)
    DevBuf r_keep, r_lo, r_hi, r_ki, r_oo, r_os, r_oq, d_gather;
    const int64_t *r_off = nullptr;
    int64_t r_n = 0, r_nkept = 0, r_total = 0;
    bool r_gathered = false, r_gathered_qual = false;
    // caller-supplied bytes staged for the length of one call (records of itsx_trim_*, sequences of itsx_search_seqs, chunk
    // offsets of itsx_reads_append): apart from d_ascii / d_off / d_qual so that the resident reads survive
    DevBuf d_stage_seq, d_stage_qual, d_stage_off;

    // one sample sharded over G GPUs (shard.cu): bucket order of the block's uniques, scratch, send / receive staging
    int sh_G = 0;
    int64_t sh_bytes = 0;
    DevBuf d_sh_order, d_sh_tmp, d_sh_bases, d_sh_rec;

    std::vector<cudaStream_t> lanes;      // side streams for the per-profile launches
    std::vector<cudaEvent_t> lane_ev;     // ordering-only events: one per lane, and lane_fork on c->stream
    cudaEvent_t lane_fork = nullptr;
};

enum { CNT_COLLIDE = 0, CNT_PAST_FWD, CNT_FWD_ROWS, CNT_BCK_ROWS, CNT_ENV_ROWS, CNT_DOM_OVERFLOW, CNT_MULTI,
       CNT_HITS_REPORTED, CNT_DOM_REPORTED, CNT_MAX_ENVLEN, CNT_BIAS_ROWS, CNT_NDOM, CNT_SEL_MULTI, CNT_CERTAIN, CNT_VIT_ROWS, CNT_VIT_RUN, CNT_N };

#define CUDA_TRY(ctx, call)                                                                   \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e__);                 \
            return ITSX_ECUDA;                                                                \
        }                                                                                     \
    } while (0)

// CUB's two-call temp-storage protocol for one or more operations queued back to back on c->d_tmp.  Each f is a callable
// (void *tmp, size_t &bytes) -> cudaError_t around one CUB call.  Every f is sized before d_tmp grows, once: growing it
// between two of them would free storage that the first, already queued, still uses.  Returns the first failure.
template <typename... F>
cudaError_t cub_run(itsx_ctx *c, F &&...f)
{
    size_t bytes[sizeof...(F)] = {}, need = 0;
    cudaError_t e = cudaSuccess;
    int i = 0;
    auto size = [&](auto &g) { if (e == cudaSuccess) { e = g(nullptr, bytes[i]); need = std::max(need, bytes[i]); } i++; };
    (size(f), ...);
    if (e == cudaSuccess) e = c->d_tmp.ensure(need);
    i = 0;
    auto run = [&](auto &g) { if (e == cudaSuccess) e = g(c->d_tmp.p, bytes[i]); i++; };
    (run(f), ...);
    return e;
}

// fan-out of c->stream to the side streams lanes[0 .. n) (ensure_lanes creates them), and fan-in back to c->stream
inline cudaError_t fork_lanes(itsx_ctx *c, int n)
{
    cudaError_t e = cudaEventRecord(c->lane_fork, c->stream);
    for (int l = 0; l < n && e == cudaSuccess; l++) e = cudaStreamWaitEvent(c->lanes[l], c->lane_fork, 0);
    return e;
}
inline cudaError_t join_lanes(itsx_ctx *c, int n)
{
    cudaError_t e = cudaSuccess;
    for (int l = 0; l < n && e == cudaSuccess; l++) {
        e = cudaEventRecord(c->lane_ev[l], c->lanes[l]);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(c->stream, c->lane_ev[l], 0);
    }
    return e;
}

// N timing events, destroyed with the set; ms(i, j) is the time from event i to event j, 0 if either is not complete
template <int N>
struct Timeline {
    cudaEvent_t ev[N] = {};
    cudaError_t status = cudaSuccess;     // of the creation
    Timeline() { for (auto &e : ev) if (status == cudaSuccess) status = cudaEventCreate(&e); }
    ~Timeline() { for (auto e : ev) if (e) cudaEventDestroy(e); }
    Timeline(const Timeline &) = delete;            // owns its events
    Timeline &operator=(const Timeline &) = delete;
    cudaError_t record(int i, cudaStream_t st) const { return cudaEventRecord(ev[i], st); }
    float ms(int i, int j) const { float t = 0.f; cudaEventElapsedTime(&t, ev[i], ev[j]); return t; }
};

#ifdef __CUDACC__
// byte mover of the trim / re-expansion and shard-exchange kernels: segment j = src[soff[j] .. + len) -> dst[doff[j] ..), one group of
// `width` lanes (a warp, or 8 lanes for slices of ~130 bytes) per segment,
// 16-byte stores on the aligned middle of the destination, bytes at its head and tail.  Source words are read as
// aligned 32-bit words and funnel-shifted into place, so neither side needs any alignment.
__device__ __forceinline__ void group_copy(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int n, int lane,
                                           int width)
{
    const int head = min(n, (int)((16 - ((uintptr_t)dst & 15)) & 15));
    for (int b = lane; b < head; b += width) dst[b] = src[b];
    const int nvec = (n - head) >> 4;
    const uint8_t *s = src + head;
    uint4 *d4 = (uint4 *)(dst + head);
    const int sh = (int)((uintptr_t)s & 3) * 8;
    const uint32_t *sw = (const uint32_t *)((uintptr_t)s & ~(uintptr_t)3);
    for (int v = lane; v < nvec; v += width) {
        const uint32_t *p = sw + v * 4;
        const uint32_t w0 = p[0], w1 = p[1], w2 = p[2], w3 = p[3];
        uint4 o;
        if (sh == 0) {
            o = make_uint4(w0, w1, w2, w3);
        } else {
            const uint32_t w4 = p[4];
            o.x = __funnelshift_r(w0, w1, sh); o.y = __funnelshift_r(w1, w2, sh);
            o.z = __funnelshift_r(w2, w3, sh); o.w = __funnelshift_r(w3, w4, sh);
        }
        d4[v] = o;
    }
    const int done = head + (nvec << 4);
    for (int b = done + lane; b < n; b += width) dst[b] = src[b];
}
__device__ __forceinline__ void warp_copy(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int n, int lane)
{
    group_copy(src, dst, n, lane, 32);
}
#endif

// rows of the position table the resident read -> row map (d_uid) points into: centroids after itsx_cluster, else classes
inline int64_t map_rows(const itsx_ctx *c) { return c->cl_active ? c->cl_ncent : c->n_unique; }

// a new read set (nreads reads, total_bases bases) replaces the resident one: nothing derived from the old set stays valid
// -- derep, clustering, positions, qualities, trim output, sample ids, an open streamed upload
inline void reset_reads(itsx_ctx *c, int64_t nreads, int64_t total_bases)
{
    c->nreads = nreads;
    c->total_bases = total_bases;
    c->n_unique = 0;
    c->cl_active = false;
    c->map_external = false;
    c->pos_valid = false;
    c->qual_resident = false;
    c->r_gathered = false;
    c->have_samples = false;
    c->n_samples = 1;
    c->stream_open = false;
}

// bytes of a caller buffer (host or device) -> b, grown to bytes + pad, on c->stream
inline cudaError_t stage(itsx_ctx *c, DevBuf &b, const void *src, size_t bytes, size_t pad)
{
    cudaError_t e = b.ensure(bytes + pad);
    if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyDefault, c->stream);
    return e;
}

// stage entry points (implemented in derep.cu / search.cu / trim.cu / cluster.cu)
int derep_run(itsx_ctx *c);                                   // reads already in d_ascii/d_off
int cluster_run(itsx_ctx *c, const itsx_cluster_params *prm, const int32_t *order, int64_t *n_centroids);
void cluster_dtable(double id, int32_t lmax, int32_t *D);
int search_build_seqs_from_reads(itsx_ctx *c, const int32_t *d_first, int64_t nseq);   // resident reads d_first[0..nseq)
int search_upload_profiles(itsx_ctx *c);
int search_build_seqs_from_derep(itsx_ctx *c);                // uniques -> d_seqw
int search_build_seqs_from_host(itsx_ctx *c, const uint8_t *seq, const int64_t *off, int64_t nseq);
int search_stage1(itsx_ctx *c);
int search_stage2(itsx_ctx *c);
// trim: bounds of the reads [first, first + count) -- d_off: offsets of caller-staged records, nullptr: the resident
// reads -- into r_keep / r_lo / r_hi, r_nkept and r_total (one host synchronisation); then the re-expansion of their kept
// slices of d_seq / d_qual (nullptr: bases only) into r_ki / r_oo / r_os / r_oq; trim_fetch_dev queues the copy of that
// re-expansion to caller buffers (any may be NULL; the caller synchronises)
int trim_bounds_dev(itsx_ctx *c, int mode, const int64_t *d_off, int64_t first, int64_t count);
int trim_gather_dev(itsx_ctx *c, const uint8_t *d_seq, const uint8_t *d_qual);
int trim_fetch_dev(itsx_ctx *c, int32_t *kept_index, int64_t *out_off, uint8_t *out_seq, uint8_t *out_qual);
