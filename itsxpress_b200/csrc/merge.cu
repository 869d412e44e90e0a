// merge.cu -- paired-end read merging on the GPU: the step in front of dereplication for paired input.
//
// Replaces the `vsearch --fastq_mergepairs R1 --reverse R2 --fastqout seq.fq --fastq_maxdiffs 40 --fastq_maxee 2
// [--fastq_allowmergestagger] --fastq_qmax 93` process of SeqSamplePairedNotInterleaved._merge_reads
// (itsxpress/SeqSample.py:266-365, argv :314-349; constants definitions.py:79,82).  SURVEY section 8(f) row 2.
// Same decisions and the same bytes as oracle/ora_merge.c (which states the algorithm and its provenance).
//
// One warp per pair, reads staged in shared memory:
//   * candidate diagonals ("at least four matching 5-mers"): the reads are turned into four bit planes (A, C, G, T;
//     one bit per base, built with warp ballots); for a diagonal the forward planes are ANDed with the funnel-shifted
//     planes of the reverse complement, and the 5-mer hits are  m & m>>1 & m>>2 & m>>3 & m>>4  counted with popc:
//     32 bases per instruction instead of a byte compare per cell.  Lanes stride over the F + R - 1 diagonals.
//     Lanes take 32 consecutive diagonals at a time.
//   * the candidates of a group are scored one after the other by the whole warp: lanes fetch bases, qualities and
//     the log-odds of 32 overlap positions in parallel, then the running sum / running maximum / drop test are
//     replayed in sequence from shared memory (double precision, from the 3' end: the summation order and the drop
//     test are part of the result).  Candidates come up in ascending offset, which is the order the
//     "first strictly greater score wins" rule needs;
//   * the merged read is written by all lanes; the expected-error sum is taken from strided partial sums unless it
//     falls within rounding distance of maxee, in which case it is replayed in read order (see there).
// HBM traffic is the reads in and the merged reads out (about 3 (F + R) bytes per pair); the kernel is bound by
// instruction issue (plane work on the integer pipe, the sequential double-precision replay).
#include <cmath>
#include <cub/cub.cuh>
#include "itsx_internal.h"

namespace {

constexpr int MG_WARPS = 4;        // pairs in flight per CTA
constexpr int MG_NQ = 94;          // quality values 0..93
constexpr int MG_MINDIAG = 4;     // a diagonal needs this many matching 5-mers to be scored

struct MergeTabs {
    double  match[MG_NQ * MG_NQ], mism[MG_NQ * MG_NQ], q2p[MG_NQ];
    uint8_t same[MG_NQ * MG_NQ], diff[MG_NQ * MG_NQ];
};

struct MergeArgs {
    const uint8_t *fseq, *fqual, *rseq, *rqual;
    const int64_t *foff, *roff;
    int64_t        npairs;
    const MergeTabs *tabs;
    int            maxdiffs, allow_stagger, qmax, minovlen, ascii;
    double         maxee, maxdiffpct;
    int            WF, WR, LF, LR;           // words per plane, padded byte lengths (shared-memory layout)
    int32_t       *merged_len;
    uint8_t       *reason;
    uint8_t       *oseq, *oqual;             // slot of pair i starts at foff[i] + roff[i]
    int           *badflag;
    unsigned long long *hist;                // [16] pairs per reason
};

__device__ __forceinline__ uint8_t mg_up(uint8_t c) { return (c >= 'a' && c <= 'z') ? (uint8_t)(c - 32) : c; }
__device__ __forceinline__ uint8_t mg_comp(uint8_t c)
{
    switch (c) {
    case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'T': return 'A'; case 'U': return 'A';
    case 'R': return 'Y'; case 'Y': return 'R'; case 'S': return 'S'; case 'W': return 'W'; case 'K': return 'M';
    case 'M': return 'K'; case 'B': return 'V'; case 'D': return 'H'; case 'H': return 'D'; case 'V': return 'B';
    default:  return 'N';
    }
}

__global__ void __launch_bounds__(MG_WARPS * 32) merge_kernel(const MergeArgs a)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ double s_q2p[MG_NQ];
    for (int t = threadIdx.x; t < MG_NQ; t += blockDim.x) s_q2p[t] = a.tabs->q2p[t];
    __syncthreads();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const size_t per_warp = (size_t)16 * (a.WF + a.WR + 2) + (size_t)3 * (a.LF + a.LR);
    unsigned char *base = smem + per_warp * wib;
    // rc planes carry one zero word in front and one behind the data (the shifted reads of a diagonal reach word
    // -1 and word nwR, never further), so the diagonal loop needs no bounds checks
    const int SR = a.WR + 2;
    uint32_t *PF = (uint32_t *)base, *PR = PF + 4 * a.WF;
    uint8_t *fs = (uint8_t *)(PR + 4 * SR), *fq = fs + a.LF, *rc = fq + a.LF, *rcq = rc + a.LR, *mq = rcq + a.LR;
    __shared__ double s_delta[MG_WARPS][32];
    double *sd = s_delta[wib];
    const double *tmatch = a.tabs->match, *tmism = a.tabs->mism;
    const int a0 = a.ascii;

    const int64_t nwarps = (int64_t)gridDim.x * MG_WARPS;
    for (int64_t pair = (int64_t)blockIdx.x * MG_WARPS + wib; pair < a.npairs; pair += nwarps) {
        const int64_t fo = a.foff[pair], ro = a.roff[pair];
        const int F = (int)(a.foff[pair + 1] - fo), R = (int)(a.roff[pair + 1] - ro);
        __syncwarp();
        bool bad = false;
        for (int p = lane; p < F; p += 32) {
            const uint8_t q = a.fqual[fo + p];
            fs[p] = mg_up(a.fseq[fo + p]);
            fq[p] = q;
            bad |= (int)q - a0 < 0 || (int)q - a0 > a.qmax;
        }
        for (int p = lane; p < R; p += 32) {
            const uint8_t q = a.rqual[ro + R - 1 - p];
            rc[p] = mg_comp(mg_up(a.rseq[ro + R - 1 - p]));
            rcq[p] = q;
            bad |= (int)q - a0 < 0 || (int)q - a0 > a.qmax;
        }
        __syncwarp();
        if (__any_sync(0xffffffffu, bad)) {       // vsearch stops with a fatal error; the host turns the flag into one
            if (lane == 0) {
                a.merged_len[pair] = 0;
                a.reason[pair] = ITSX_MERGE_BADQUAL;
                atomicExch(a.badflag, 1);
                atomicAdd(&a.hist[ITSX_MERGE_BADQUAL], 1ull);
            }
            continue;
        }
        // bit planes
        const int nwF = (F + 31) >> 5, nwR = (R + 31) >> 5;
        for (int j = 0; j < nwF; j++) {
            const int p = 32 * j + lane;
            const uint8_t c = p < F ? fs[p] : 0;
            const uint32_t bA = __ballot_sync(0xffffffffu, c == 'A'), bC = __ballot_sync(0xffffffffu, c == 'C'),
                           bG = __ballot_sync(0xffffffffu, c == 'G'), bT = __ballot_sync(0xffffffffu, c == 'T');
            if (lane == 0) { PF[j] = bA; PF[a.WF + j] = bC; PF[2 * a.WF + j] = bG; PF[3 * a.WF + j] = bT; }
        }
        for (int j = 0; j < nwR; j++) {
            const int p = 32 * j + lane;
            const uint8_t c = p < R ? rc[p] : 0;
            const uint32_t bA = __ballot_sync(0xffffffffu, c == 'A'), bC = __ballot_sync(0xffffffffu, c == 'C'),
                           bG = __ballot_sync(0xffffffffu, c == 'G'), bT = __ballot_sync(0xffffffffu, c == 'T');
            if (lane == 0) { PR[1 + j] = bA; PR[SR + 1 + j] = bC; PR[2 * SR + 1 + j] = bG; PR[3 * SR + 1 + j] = bT; }
        }
        if (lane < 4) { PR[lane * SR] = 0u; PR[lane * SR + 1 + nwR] = 0u; }
        __syncwarp();

        // Diagonals in ascending order, 32 at a time: every lane counts the 5-mer hits of its own diagonal; the
        // candidates of the group are then scored one after the other BY THE WHOLE WARP (lanes fetch the bases,
        // qualities and table entries of 32 overlap positions in parallel; the running sum / maximum / drop logic
        // is replayed in sequence from shared memory, warp-uniformly).  Scoring order = ascending offset, so the
        // "first strictly greater score" rule needs no reduction.
        double best_score = 0.0;
        int best_i = 0, best_diffs = 0, hits = 0, kmers = 0;
        const int ndiag = F + R - 1;
        for (int gi = 1; gi <= ndiag; gi += 32) {
            const int i = gi + lane;
            int cnt = 0;
            if (i <= ndiag) {
                const int sh = F - i;                        // forward position p pairs with rc position p - sh
                const int p0 = sh > 0 ? sh : 0, p1 = F < sh + R ? F : sh + R;
                const int j0 = p0 >> 5, j1 = (p1 - 1) >> 5;
                // match word j = OR over the planes of  PF[j] & (PR >> (32 j - sh)):  the shift within a word (r) is the
                // same for every j, the rc word index q advances with j, so each rc word is loaded once and carried
                const int t0 = 32 * j0 - sh, r = t0 & 31;
                int q = t0 >> 5;
                auto rword = [&](int x, int qq) -> uint32_t { return PR[x * SR + 1 + qq]; };     // qq in [-1, nwR]
                uint32_t lo0 = rword(0, q), lo1 = rword(1, q), lo2 = rword(2, q), lo3 = rword(3, q);
                uint32_t prev = 0;
                for (int j = j0; j <= j1 + 1; j++) {
                    uint32_t m = 0;
                    if (j <= j1) {
                        const uint32_t hi0 = rword(0, q + 1), hi1 = rword(1, q + 1), hi2 = rword(2, q + 1),
                                       hi3 = rword(3, q + 1);
                        m = (PF[j] & __funnelshift_r(lo0, hi0, r)) | (PF[a.WF + j] & __funnelshift_r(lo1, hi1, r)) |
                            (PF[2 * a.WF + j] & __funnelshift_r(lo2, hi2, r)) |
                            (PF[3 * a.WF + j] & __funnelshift_r(lo3, hi3, r));
                        lo0 = hi0; lo1 = hi1; lo2 = hi2; lo3 = hi3;
                        q++;
                    }
                    if (j > j0) {           // 5-mer hits that START in word j - 1 (bits 32.. come from word j)
                        const uint32_t m5 = prev & __funnelshift_r(prev, m, 1) & __funnelshift_r(prev, m, 2) &
                                            __funnelshift_r(prev, m, 3) & __funnelshift_r(prev, m, 4);
                        cnt += __popc(m5);
                    }
                    prev = m;
                }
            }
            unsigned cand = __ballot_sync(0xffffffffu, cnt >= MG_MINDIAG);
            while (cand) {
                const int ci = gi + __ffs(cand) - 1;
                cand &= cand - 1;
                kmers = 1;
                const int sh = F - ci;
                const int p0 = sh > 0 ? sh : 0, p1 = F < sh + R ? F : sh + R;
                const int len = p1 - p0;
                double score = 0.0, high = 0.0, dropmax = 0.0;
                int diffs = 0;
                bool pend = false;
                for (int e0 = 0; e0 < len; e0 += 32) {
                    const int e = e0 + lane, p = p1 - 1 - e;      // scoring runs from the 3' end of the forward read
                    bool eq = true;
                    double d = 0.0;
                    if (e < len) {
                        const int qa = fq[p] - a0, qb = rcq[p - sh] - a0;
                        eq = fs[p] == rc[p - sh];
                        d = __ldg(eq ? &tmatch[qa * MG_NQ + qb] : &tmism[qa * MG_NQ + qb]);
                    }
                    const unsigned eqm = __ballot_sync(0xffffffffu, eq);
                    // "fast" element: a match whose log-odds are >= 0 (all but the Q < 2 corner, where rounding can
                    // leave -1e-16).  It cannot lower the score, so within a run of fast elements the running
                    // maximum only has to be taken when the run ends (pend).  Everything else is replayed literally.
                    const unsigned fastm = __ballot_sync(0xffffffffu, eq && d >= 0.0);
                    __syncwarp();
                    sd[lane] = d;
                    __syncwarp();
                    const int ne = min(32, len - e0);
                    diffs += __popc(~eqm);
                    for (int t = 0; t < ne; t++) {
                        if ((fastm >> t) & 1u) {
                            score += sd[t];
                            pend = true;
                        } else {
                            if (pend) { if (score > high) high = score; pend = false; }
                            score += sd[t];
                            if ((eqm >> t) & 1u) { if (score > high) high = score; }
                            else if (score < high - dropmax) dropmax = high - score;
                        }
                    }
                    // once the drop below the maximum has reached 16 bits the diagonal scores 0 whatever follows
                    if (dropmax >= 16.0) break;
                }
                if (dropmax >= 16.0) score = 0.0;
                if (score >= 16.0) hits++;
                if (score > best_score) { best_score = score; best_i = ci; best_diffs = diffs; }
            }
        }
        int why = ITSX_MERGE_OK;
        if (hits > 1) why = ITSX_MERGE_REPEAT;
        else if (!a.allow_stagger && best_i > F) why = ITSX_MERGE_STAGGERED;
        else if (best_diffs > a.maxdiffs) why = ITSX_MERGE_MAXDIFFS;
        else if (best_i > 0 && 100.0 * best_diffs / best_i > a.maxdiffpct) why = ITSX_MERGE_MAXDIFFPCT;
        else if (!kmers) why = ITSX_MERGE_NOKMERS;
        else if (best_score < 16.0) why = ITSX_MERGE_MINSCORE;
        else if (best_i < a.minovlen) why = ITSX_MERGE_MINOVLEN;
        int n = 0;
        if (why == ITSX_MERGE_OK) {
            const int sh = F - best_i;
            const int nA = sh > 0 ? sh : 0, r0 = sh < 0 ? -sh : 0;
            const int ov = min(F - nA, R - r0);
            n = nA + ov + (R - r0 - ov);
            const uint8_t *tsame = a.tabs->same, *tdiff = a.tabs->diff;
            const int64_t slot = fo + ro;
            double part = 0.0;
            for (int m = lane; m < n; m += 32) {
                uint8_t s, q;
                if (m < nA) { s = fs[m]; q = fq[m]; }
                else if (m < nA + ov) {
                    const uint8_t x = fs[m], y = rc[m - sh];
                    const int qa = fq[m] - a0, qb = rcq[m - sh] - a0;
                    if (y == 'N') { s = x; q = fq[m]; }
                    else if (x == 'N') { s = y; q = rcq[m - sh]; }
                    else if (x == y) { s = x; q = __ldg(&tsame[qa * MG_NQ + qb]); }
                    else if (qa > qb) { s = x; q = __ldg(&tdiff[qa * MG_NQ + qb]); }
                    else { s = y; q = __ldg(&tdiff[qb * MG_NQ + qa]); }
                } else { s = rc[m - sh]; q = rcq[m - sh]; }
                a.oseq[slot + m] = s;
                a.oqual[slot + m] = q;
                mq[m] = q;
                part += s_q2p[q - a0];
            }
            // Expected errors: the reference sums them in read order and the comparison with maxee is part of the
            // result.  A sum in any other order differs from it by less than 2 n u sum|x| (u = 2^-53; n < 2^14 here),
            // i.e. by far less than 1e-9 relative, so the strided partial sums decide unless the total lies inside
            // that band around maxee -- only then is the sum replayed in read order by one lane.
#pragma unroll
            for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
            __syncwarp();
            int ok;
            const double band = 1e-9 * (1.0 + fabs(part));
            if (part > a.maxee + band) ok = 0;
            else if (part < a.maxee - band) ok = 1;
            else {
                ok = 1;
                if (lane == 0) {
                    double ee = 0.0;
                    for (int m = 0; m < n; m++) ee += s_q2p[mq[m] - a0];
                    ok = ee <= a.maxee;
                }
                ok = __shfl_sync(0xffffffffu, ok, 0);
            }
            if (!ok) { why = ITSX_MERGE_MAXEE; n = 0; }
        }
        if (lane == 0) {
            a.merged_len[pair] = n;
            a.reason[pair] = (uint8_t)why;
            atomicAdd(&a.hist[why], 1ull);
        }
    }
}

__global__ void merge_flag_kernel(const int32_t *__restrict__ mlen, int64_t n, int32_t *__restrict__ flag,
                                  int64_t *__restrict__ len64)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    flag[i] = i < n && mlen[i] > 0;
    len64[i] = i < n ? mlen[i] : 0;
}

// one warp per pair: merged reads out of their slots into back-to-back buffers
__global__ void __launch_bounds__(256)
merge_compact_kernel(const int32_t *__restrict__ mlen, const int32_t *__restrict__ kscan, const int64_t *__restrict__ lscan,
                     const int64_t *__restrict__ foff, const int64_t *__restrict__ roff, int64_t n,
                     const uint8_t *__restrict__ sseq, const uint8_t *__restrict__ squal, int32_t *__restrict__ idx,
                     int64_t *__restrict__ ooff, uint8_t *__restrict__ oseq, uint8_t *__restrict__ oqual)
{
    const int lane = threadIdx.x & 31;
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i > n) return;
    if (i == n) { if (lane == 0) ooff[kscan[n]] = lscan[n]; return; }
    const int len = mlen[i];
    if (len <= 0) return;
    const int64_t src = foff[i] + roff[i], dst = lscan[i];
    if (lane == 0) { idx[kscan[i]] = (int32_t)i; ooff[kscan[i]] = dst; }
    for (int b = lane; b < len; b += 32) { oseq[dst + b] = sseq[src + b]; oqual[dst + b] = squal[src + b]; }
}

struct Diff {
    const int64_t *o;
    __host__ __device__ int operator()(int64_t i) const { return (int)(o[i + 1] - o[i]); }
};

inline unsigned nblk(int64_t n, int b) { return (unsigned)((n + b - 1) / b); }

double q_to_p(int x) { return x < 2 ? 0.75 : exp10(-x / 10.0); }
uint8_t q_from_p(double p, const itsx_merge_params &prm)
{
    int q = (int)std::round(-10.0 * std::log10(p));
    q = std::min(q, prm.qmaxout);
    q = std::max(q, prm.qminout);
    return (uint8_t)(prm.ascii + q);
}
// posterior qualities and overlap scores for every pair of quality values (Edgar & Flyvbjerg 2015), host libm
void make_tabs(MergeTabs &t, const itsx_merge_params &prm)
{
    for (int x = 0; x < MG_NQ; x++) {
        const double px = q_to_p(x);
        t.q2p[x] = px;
        for (int y = 0; y < MG_NQ; y++) {
            const double py = q_to_p(y);
            t.same[x * MG_NQ + y]  = q_from_p(px * py / 3.0 / (1.0 - px - py + 4.0 * px * py / 3.0), prm);
            t.diff[x * MG_NQ + y]  = q_from_p(px * (1.0 - py / 3.0) / (px + py - 4.0 * px * py / 3.0), prm);
            t.match[x * MG_NQ + y] = std::log2((1.0 - px - py + px * py * 4.0 / 3.0) / 0.25);
            t.mism[x * MG_NQ + y]  = std::log2(((px + py) / 3.0 - px * py * 4.0 / 9.0) / 0.25);
        }
    }
}

}  // namespace

extern "C" {

void itsx_merge_default_params(itsx_merge_params *p)
{
    if (!p) return;
    p->maxdiffs = 40; p->allow_stagger = 0; p->qmax = 93;
    p->minovlen = 10; p->qmaxout = 41; p->qminout = 0; p->ascii = 33; p->reserved = 0;
    p->maxee = 2.0; p->maxdiffpct = 100.0;
}

int itsx_merge_pairs(itsx_ctx *c, const uint8_t *fseq, const uint8_t *fqual, const int64_t *foff, const uint8_t *rseq,
                     const uint8_t *rqual, const int64_t *roff, int64_t npairs, const itsx_merge_params *prm,
                     int32_t *merged_len, uint8_t *reason, int64_t *n_merged, int64_t *total)
{
    if (!c) return ITSX_EINVAL;
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (npairs < 0 || !foff || !roff || (npairs > 0 && (!fseq || !fqual || !rseq || !rqual))) {
        c->err = "merge: null input";
        return ITSX_EINVAL;
    }
    itsx_merge_params p;
    if (prm) p = *prm; else itsx_merge_default_params(&p);
    if (p.qmax < 0 || p.qmax >= MG_NQ || p.ascii < 0 || p.ascii + MG_NQ > 256 || p.qmaxout >= MG_NQ || p.qminout < 0) {
        c->err = "merge: quality range must lie within 0..93";
        return ITSX_EINVAL;
    }
    cudaStream_t st = c->stream;
    c->mg_npairs = npairs;
    c->mg_nmerged = 0;
    c->mg_total = 0;
    c->mgstats = itsx_merge_stats{};
    c->mgstats.n_pairs = npairs;
    if (n_merged) *n_merged = 0;
    if (total) *total = 0;
    if (npairs == 0) return ITSX_OK;
    if (npairs > INT32_MAX - 1) { c->err = "merge: more than 2^31 pairs in one call"; return ITSX_ELIMIT; }
    Timeline<2> tl;     // merge_kernel alone
    CUDA_TRY(c, tl.status);

    const int64_t ftot = itsx_peek_i64(foff + npairs), rtot = itsx_peek_i64(roff + npairs);
    CUDA_TRY(c, c->d_mg_foff.ensure((size_t)(npairs + 1) * 8));
    CUDA_TRY(c, c->d_mg_roff.ensure((size_t)(npairs + 1) * 8));
    CUDA_TRY(c, c->d_mg_fseq.ensure((size_t)ftot + 16));
    CUDA_TRY(c, c->d_mg_fqual.ensure((size_t)ftot + 16));
    CUDA_TRY(c, c->d_mg_rseq.ensure((size_t)rtot + 16));
    CUDA_TRY(c, c->d_mg_rqual.ensure((size_t)rtot + 16));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_mg_foff.p, foff, (size_t)(npairs + 1) * 8, cudaMemcpyDefault, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_mg_roff.p, roff, (size_t)(npairs + 1) * 8, cudaMemcpyDefault, st));
    if (ftot) {
        CUDA_TRY(c, cudaMemcpyAsync(c->d_mg_fseq.p, fseq, (size_t)ftot, cudaMemcpyDefault, st));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_mg_fqual.p, fqual, (size_t)ftot, cudaMemcpyDefault, st));
    }
    if (rtot) {
        CUDA_TRY(c, cudaMemcpyAsync(c->d_mg_rseq.p, rseq, (size_t)rtot, cudaMemcpyDefault, st));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_mg_rqual.p, rqual, (size_t)rtot, cudaMemcpyDefault, st));
    }
    // longest reads decide the shared-memory layout
    CUDA_TRY(c, c->d_mg_len64.ensure((size_t)(npairs + 1) * 8));
    CUDA_TRY(c, c->d_mg_flag.ensure((size_t)(npairs + 1) * 4));
    CUDA_TRY(c, c->d_mg_kscan.ensure((size_t)(npairs + 1) * 4));
    CUDA_TRY(c, c->d_mg_lscan.ensure((size_t)(npairs + 1) * 8));
    int maxF = 0, maxR = 0;
    {
        // adjacent differences + max, on the device (cub transform iterators would do; two tiny reductions suffice)
        cub::CountingInputIterator<int64_t> cnt(0);
        cub::TransformInputIterator<int, Diff, cub::CountingInputIterator<int64_t>> itF(cnt, Diff{c->d_mg_foff.as<int64_t>()}),
            itR(cnt, Diff{c->d_mg_roff.as<int64_t>()});
        int *d_max = (int *)c->d_mg_kscan.p;
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceReduce::Max(t, b, itF, d_max, (int)npairs, st); },
                            [&](void *t, size_t &b) { return cub::DeviceReduce::Max(t, b, itR, d_max + 1, (int)npairs, st); }));
        c->launches += 2;
        int h[2] = {0, 0};
        CUDA_TRY(c, cudaMemcpyAsync(h, d_max, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        maxF = h[0];
        maxR = h[1];
    }
    if (maxF < 0 || maxR < 0) { c->err = "merge: offsets must ascend"; return ITSX_EINVAL; }
    MergeArgs a{};
    a.WF = std::max(1, (maxF + 31) / 32);
    a.WR = std::max(1, (maxR + 31) / 32);
    a.LF = (maxF + 3) & ~3;
    a.LR = (maxR + 3) & ~3;
    const size_t per_warp = (size_t)16 * (a.WF + a.WR + 2) + (size_t)3 * (a.LF + a.LR);
    const size_t smem = per_warp * MG_WARPS;
    if (smem > 200 * 1024) {
        c->err = "merge: reads longer than the shared-memory staging allows (" + std::to_string(maxF) + " + " +
                 std::to_string(maxR) + " bases)";
        return ITSX_ELIMIT;
    }
    // tables
    if (!c->mg_tabs_ready || std::memcmp(&c->mg_tabs_prm, &p, sizeof p) != 0) {
        static thread_local MergeTabs h_tabs;
        make_tabs(h_tabs, p);
        CUDA_TRY(c, c->d_mg_tabs.ensure(sizeof(MergeTabs)));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_mg_tabs.p, &h_tabs, sizeof(MergeTabs), cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        c->mg_tabs_prm = p;
        c->mg_tabs_ready = true;
    }
    CUDA_TRY(c, c->d_mg_mlen.ensure((size_t)npairs * 4 + 16));
    CUDA_TRY(c, c->d_mg_reason.ensure((size_t)npairs + 16));
    CUDA_TRY(c, c->d_mg_sseq.ensure((size_t)(ftot + rtot) + 16));
    CUDA_TRY(c, c->d_mg_squal.ensure((size_t)(ftot + rtot) + 16));
    CUDA_TRY(c, c->d_mg_hist.ensure(17 * 8));
    CUDA_TRY(c, cudaMemsetAsync(c->d_mg_hist.p, 0, 17 * 8, st));
    a.fseq = c->d_mg_fseq.as<uint8_t>(); a.fqual = c->d_mg_fqual.as<uint8_t>();
    a.rseq = c->d_mg_rseq.as<uint8_t>(); a.rqual = c->d_mg_rqual.as<uint8_t>();
    a.foff = c->d_mg_foff.as<int64_t>(); a.roff = c->d_mg_roff.as<int64_t>();
    a.npairs = npairs;
    a.tabs = c->d_mg_tabs.as<MergeTabs>();
    a.maxdiffs = p.maxdiffs; a.allow_stagger = p.allow_stagger; a.qmax = p.qmax; a.minovlen = p.minovlen; a.ascii = p.ascii;
    a.maxee = p.maxee; a.maxdiffpct = p.maxdiffpct;
    a.merged_len = c->d_mg_mlen.as<int32_t>();
    a.reason = c->d_mg_reason.as<uint8_t>();
    a.oseq = c->d_mg_sseq.as<uint8_t>(); a.oqual = c->d_mg_squal.as<uint8_t>();
    a.hist = c->d_mg_hist.as<unsigned long long>();
    a.badflag = (int *)(a.hist + 16);
    CUDA_TRY(c, cudaFuncSetAttribute(merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CUDA_TRY(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, merge_kernel, MG_WARPS * 32, smem));
    per_sm = std::max(per_sm, 1);
    const int64_t want = (npairs + MG_WARPS - 1) / MG_WARPS;
    const unsigned grid = (unsigned)std::min<int64_t>(want, (int64_t)c->sm_count * per_sm);   // persistent: whole waves of resident CTAs
    CUDA_TRY(c, tl.record(0, st));
    merge_kernel<<<grid, MG_WARPS * 32, smem, st>>>(a);
    CUDA_TRY(c, tl.record(1, st));
    // compaction: merged pairs in input order, back to back
    int32_t *flag = c->d_mg_flag.as<int32_t>(), *ks = c->d_mg_kscan.as<int32_t>();
    int64_t *l64 = c->d_mg_len64.as<int64_t>(), *ls = c->d_mg_lscan.as<int64_t>();
    merge_flag_kernel<<<nblk(npairs + 1, 256), 256, 0, st>>>(a.merged_len, npairs, flag, l64);
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, flag, ks, (int)npairs + 1, st); },
                        [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, l64, ls, (int)npairs + 1, st); }));
    c->launches += 4;
    int32_t nk = 0;
    int64_t tot = 0;
    unsigned long long hist[17];
    CUDA_TRY(c, cudaMemcpyAsync(&nk, ks + npairs, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaMemcpyAsync(&tot, ls + npairs, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaMemcpyAsync(hist, c->d_mg_hist.p, sizeof hist, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, c->d_mg_idx.ensure((size_t)std::max(nk, 1) * 4));
    CUDA_TRY(c, c->d_mg_ooff.ensure((size_t)(nk + 1) * 8));
    CUDA_TRY(c, c->d_mg_oseq.ensure((size_t)std::max<int64_t>(tot, 1)));
    CUDA_TRY(c, c->d_mg_oqual.ensure((size_t)std::max<int64_t>(tot, 1)));
    merge_compact_kernel<<<nblk((npairs + 1) * 32, 256), 256, 0, st>>>(a.merged_len, ks, ls, a.foff, a.roff, npairs, a.oseq,
                                                                       a.oqual, c->d_mg_idx.as<int32_t>(),
                                                                       c->d_mg_ooff.as<int64_t>(), c->d_mg_oseq.as<uint8_t>(),
                                                                       c->d_mg_oqual.as<uint8_t>());
    c->launches += 1;
    if (merged_len) CUDA_TRY(c, cudaMemcpyAsync(merged_len, a.merged_len, (size_t)npairs * 4, cudaMemcpyDefault, st));
    if (reason) CUDA_TRY(c, cudaMemcpyAsync(reason, a.reason, (size_t)npairs, cudaMemcpyDefault, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    c->mg_nmerged = nk;
    c->mg_total = tot;
    c->mgstats.n_merged = nk;
    c->mgstats.bytes_in = 2 * (ftot + rtot);
    c->mgstats.bytes_out = 2 * tot;
    c->mgstats.ms_kernel = tl.ms(0, 1);
    for (int r = 0; r < 16; r++) c->mgstats.by_reason[r] = (int64_t)hist[r];
    if (n_merged) *n_merged = nk;
    if (total) *total = tot;
    if (hist[16]) {
        c->err = "merge: FASTQ quality value outside [0, " + std::to_string(p.qmax) + "] (--fastq_qmax)";
        return ITSX_EFORMAT;
    }
    return ITSX_OK;
}

int itsx_merge_fetch(itsx_ctx *c, int32_t *merged_index, int64_t *out_off, uint8_t *out_seq, uint8_t *out_qual)
{
    if (!c) return ITSX_EINVAL;
    CUDA_TRY(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int64_t nk = c->mg_nmerged, tot = c->mg_total;
    if (c->mg_npairs == 0 || nk == 0) {
        if (out_off) { const int64_t z = 0; CUDA_TRY(c, cudaMemcpyAsync(out_off, &z, 8, cudaMemcpyDefault, st)); }
        CUDA_TRY(c, cudaStreamSynchronize(st));
        return ITSX_OK;
    }
    if (merged_index) CUDA_TRY(c, cudaMemcpyAsync(merged_index, c->d_mg_idx.p, (size_t)nk * 4, cudaMemcpyDefault, st));
    if (out_off) CUDA_TRY(c, cudaMemcpyAsync(out_off, c->d_mg_ooff.p, (size_t)(nk + 1) * 8, cudaMemcpyDefault, st));
    if (out_seq && tot) CUDA_TRY(c, cudaMemcpyAsync(out_seq, c->d_mg_oseq.p, (size_t)tot, cudaMemcpyDefault, st));
    if (out_qual && tot) CUDA_TRY(c, cudaMemcpyAsync(out_qual, c->d_mg_oqual.p, (size_t)tot, cudaMemcpyDefault, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return ITSX_OK;
}

int itsx_merge_get_stats(const itsx_ctx *c, itsx_merge_stats *s)
{
    if (!c || !s) return ITSX_EINVAL;
    *s = c->mgstats;
    return ITSX_OK;
}

}  // extern "C"
