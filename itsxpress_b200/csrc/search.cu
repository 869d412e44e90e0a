// search.cu -- profile-HMM search cascade on the GPU.
//
// Replaces `hmmsearch --domtblout -T 10 --F1 1e-6 --F2 1e-6 --F3 1e-6 --tformat fasta <hmm> rep.fa`
// (reference call site itsxpress/SeqSample.py:178-225, argv :191-209) and ItsPosition's best-boundary
// selection over the resulting table (SeqSample.py:400-429, 463-498).  Algorithm: SURVEY.md
// Appendix A (HMMER3 acceleration pipeline restated).
//
// Mapping.  Every profile in ITSx_db has M <= 45 match states, so one (sequence, profile) comparison
// is small: a whole DP row lives in ONE thread's registers.  All DP kernels are therefore
// thread-per-pair with fully unrolled node loops -- no shuffles, no shared-memory DP rows:
//   msv_kernel    u8-range MSV filter in s16x2 lanes (VIADDMNMX / VIMNMX3 DPX instructions), cost
//                 tables of a tile of profiles staged once in shared memory, grid = sequence blocks x
//                 profile tiles.  Integer-ALU bound.
//   bias_kernel   2-state composition-bias Forward on MSV survivors.
//   fb_kernel     fp32 Forward -> F3 test -> Backward -> posterior decoding -> region/envelope
//                 definition, one launch per profile so that the transition coefficients are a
//                 __grid_constant__ argument: every FFMA takes its coefficient from the constant bank
//                 and the inner loop has no load except the per-residue emission (shared memory).
//                 Parser specials go to a per-resident-warp scratch slab that stays in L2.
//   env_kernel    unihit Forward/Backward/decoding of each envelope, null2 by expectation.
//   final_kernel  per-hit and per-domain bit scores, P-values, -T threshold, reported-hit counts.
//   select/best   domE threshold with the global domZ, ItsPosition arg-max per (sequence, side).
// Floating-point order follows oracle/ora_hmm.c operation for operation (explicit fmaf, -fmad=false)
// so that envelope coordinates -- thresholded fp32 posteriors -- are reproduced exactly.
#include <cub/cub.cuh>
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include "itsx_internal.h"

namespace {

constexpr int MAXM = ITSX_MAXM;
constexpr int KP = ITSX_KP;
constexpr int MSV_TP = 32;                 // profiles per MSV tile (32 * 2 layouts * 23 * 16 * 4 B = 94 KB smem)
constexpr int MSV_THREADS = 256;           // 2 CTAs / SM by shared memory -> 16 warps / SM
constexpr int MSV_TABW = 2 * KP * 16;      // table words per profile: layout A then layout B
constexpr int FB_THREADS = 64;              // 2 warps / CTA: 6 CTAs (12 warps) per SM at 168 registers
constexpr int FB_CTAS_PER_SM = 6;
constexpr int ENV_THREADS = 128;
constexpr int ENV_CTAS_PER_SM = 2;
constexpr int SPEC_C = 5;                  // parser specials kept per row
constexpr int ENV_ROWF = MAXM + 1;             // floats per envelope row: M[1..45] (cols 0..44), Eraw (col 45)
constexpr int ENV_ROWBYTES = ENV_ROWF * 32 * 4;    // one row of one warp: 5 888 B, contiguous
constexpr int ENV_RING = 2;                    // rows of the Backward read-back ring per warp (a power of two; 4 measured slower)
// The parser specials (d_spec) and the envelope rows (d_envscratch) are sized by the longest searched sequence: about
// 18 MB and 56 MB per residue at full occupancy, so one read of a few kb would ask for more HBM than the GPU has.  Each
// buffer is held to a byte budget by running fewer tiles / warps per launch when the sequences are long; neither
// budget binds below ~600 bp, so short-read samples keep their full occupancy.
constexpr size_t FB_SCRATCH_BUDGET = (size_t)16 << 30;
constexpr size_t ENV_SCRATCH_BUDGET = (size_t)32 << 30;
static_assert((ENV_RING & (ENV_RING - 1)) == 0 && ENV_RING >= 2, "ring depth");
constexpr double kLn2 = 0.69314718055994529;
constexpr int ESTRIDE = 52;                // floats per residue row of the shared emission table (48 used)
// e_k of residue row `er` (float4 view): one 128-bit shared load serves nodes 4q .. 4q+3
#define EMIS(er, k) (((k) & 3) == 0 ? (er)[(k) >> 2].x : ((k) & 3) == 1 ? (er)[(k) >> 2].y : ((k) & 3) == 2 ? (er)[(k) >> 2].z : (er)[(k) >> 2].w)

inline unsigned nblk(int64_t n, int b) { return (unsigned)((n + b - 1) / b); }

// ------------------------------------------------------------------------------------------------
// statistics (Easel esl_gumbel_surv / esl_exp_surv / esl_exp_logsurv)
__device__ __forceinline__ double gumbel_surv(double x, double mu, double lambda)
{
    double y = lambda * (x - mu);
    double ey = -exp(-y);
    if (fabs(ey) < 5e-9) return -ey;
    return 1 - exp(ey);
}
__device__ __forceinline__ double exp_surv(double x, double mu, double lambda)
{
    if (x < mu) return 1.0;
    return exp(-lambda * (x - mu));
}
__device__ __forceinline__ double exp_logsurv(double x, double mu, double lambda)
{
    if (x < mu) return 0.0;
    return -lambda * (x - mu);
}
__device__ __forceinline__ float flogsum(const float *__restrict__ tbl, float a, float b)
{
    const float mx = a > b ? a : b, mn = a > b ? b : a;
    return (mn == -INFINITY || (mx - mn) >= 15.7f) ? mx : mx + tbl[(int)((mx - mn) * 1000.0f)];
}
__device__ __forceinline__ float logf_via_double(float x) { return (float)log((double)x); }

// residue i (0-based) of a nibble-coded sequence
__device__ __forceinline__ uint32_t residue_at(const uint32_t *__restrict__ w, int pos)
{
    return (w[pos >> 3] >> ((pos & 7) * 4)) & 15u;
}

// ------------------------------------------------------------------------------------------------
// sequence store: ASCII -> nibble codes, one warp per sequence
__global__ void seqlen_kernel(const int64_t *__restrict__ off, const int32_t *__restrict__ first, int64_t nseq,
                              int32_t *__restrict__ len, int64_t *__restrict__ nwords)
{
    int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= nseq) return;
    int64_t r = first ? first[u] : u;
    int L = (int)(off[r + 1] - off[r]);
    len[u] = L;
    nwords[u] = (L + 7) >> 3;
}
__global__ void __launch_bounds__(256) seqcode_kernel(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ off,
                                                      const int32_t *__restrict__ first, int64_t nseq,
                                                      const int64_t *__restrict__ woff, const uint8_t *__restrict__ lut,
                                                      uint32_t *__restrict__ seqw)
{
    __shared__ uint8_t s_lut[256];
    s_lut[threadIdx.x] = lut[threadIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (u >= nseq) return;
    int64_t r = first ? first[u] : u;
    const uint8_t *s = ascii + off[r];
    const int L = (int)(off[r + 1] - off[r]);
    const int nw = (L + 7) >> 3;
    uint32_t *out = seqw + woff[u];
    for (int j = lane; j < nw; j += 32) {
        uint32_t w = 0;
#pragma unroll
        for (int t = 0; t < 8; t++) {
            int p = j * 8 + t;
            uint32_t code = p < L ? s_lut[s[p]] : 0u;
            w |= code << (4 * t);
        }
        out[j] = w;
    }
}

__global__ void seqsample_kernel(const int32_t *__restrict__ sample, const int32_t *__restrict__ first, int64_t nseq,
                                 int32_t *__restrict__ out)
{
    int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < nseq) out[u] = sample[first[u]];
}

// ------------------------------------------------------------------------------------------------
// K4: MSV filter.  u8-range scores in s16x2 lanes (HMMER's u8 values; before the overflow test fires no lane can
// reach 255 - bias, so the u8 upper clamp never binds and  sv = max(max(M_{k-1}(i-1), xB) + (bias - cost), 0)
// is exact).  The diagonal dependency M_k(i) <- M_{k-1}(i-1) is absorbed by alternating two word layouts instead
// of shifting lanes every row:
//   layout A: word j = nodes (2j+1, 2j+2)      layout B: word j = nodes (2j, 2j+1)     (node 0 / 46: neutral 0)
//   A -> B:  new[j] = F(old[j-1], costB[j][x])        B -> A:  new[j] = F(old[j], costA[j][x])
// so a cell pair costs VIMNMX (xB) + VIADDMNMX (score, floor 0) + half a VIMNMX3 (row maximum) + one LDS.
__global__ void __launch_bounds__(MSV_THREADS, 2)
msv_kernel(const uint32_t *__restrict__ seqw, const int64_t *__restrict__ woff, const int32_t *__restrict__ seqlen,
           const int32_t *__restrict__ order, int64_t s0, int ns, const uint32_t *__restrict__ msvtab, const ProfScalars *__restrict__ pscal, int P,
           const uint8_t *__restrict__ tjbtab, const float *__restrict__ nullsctab, double F1,
           uint8_t *__restrict__ res, uint8_t *__restrict__ flag)
{
    extern __shared__ uint32_t s_tab[];    // [tile profiles][layout A | layout B][KP][16]
    const int p0 = blockIdx.y * MSV_TP;
    const int np = min(MSV_TP, P - p0);
    for (int t = threadIdx.x; t < np * MSV_TABW; t += MSV_THREADS) s_tab[t] = msvtab[(size_t)p0 * MSV_TABW + t];
    __syncthreads();

    const int sl = blockIdx.x * MSV_THREADS + threadIdx.x;
    const bool valid = sl < ns;
    const int64_t s = order[s0 + (valid ? sl : 0)];     // sequences are visited in order of length
    const int L = valid ? seqlen[s] : 0;
    const uint32_t *w = seqw + woff[s];
    int Lw = L;
#pragma unroll
    for (int o = 16; o; o >>= 1) Lw = max(Lw, __shfl_xor_sync(0xffffffffu, Lw, o));
    const int tjb = tjbtab[L];
    const float nullsc = nullsctab[L];

    for (int pl = 0; pl < np; pl++) {
        const ProfScalars &ps = pscal[p0 + pl];
        const int bias = ps.bias, base = ps.base, tec = ps.tec;
        const int tjbm = (tjb + ps.tbm) & 255;
        const int limit = 255 - bias;
        // the floor operand of VIADDMNMX as a run-time register (pad0 is always 0): a literal 0 makes ptxas
        // re-materialise zero registers (PRMT / IMAD.MOV) once per cell pair
        const uint32_t zero = (uint32_t)ps.pad0;
        const uint32_t *tabA = s_tab + pl * MSV_TABW, *tabB = tabA + KP * 16;
        uint32_t st[KP];
#pragma unroll
        for (int j = 0; j < KP; j++) st[j] = 0u;
        int xJ = 0, xB = max(base - tjbm, 0), resJ = 0;
        bool ovf = false;
        uint32_t wnext = L > 0 ? w[0] : 0u;
        for (int wi = 0; wi * 8 < Lw; wi++) {
            uint32_t word = wnext;
            wnext = ((wi + 1) * 8 < L) ? w[wi + 1] : 0u;       // next residue word, one block ahead
#pragma unroll
            for (int r = 0; r < 8; r++) {
                const int i = wi * 8 + r;
                const uint32_t x = word & 15u;
                word >>= 4;
                const uint32_t xB2 = (uint32_t)xB * 0x00010001u;
                if ((r & 1) == 0) {                    // layout A -> B
                    const uint32_t *tx = tabB + x;
#pragma unroll
                    for (int j = KP - 1; j >= 1; j--) st[j] = __viaddmax_s16x2(__vmaxs2(st[j - 1], xB2), tx[j * 16], zero);
                    st[0] = __viaddmax_s16x2(xB2, tx[0], zero);          // nodes (0, 1): predecessors are empty
                } else {                               // layout B -> A
                    const uint32_t *tx = tabA + x;
#pragma unroll
                    for (int j = 0; j < KP; j++) st[j] = __viaddmax_s16x2(__vmaxs2(st[j], xB2), tx[j * 16], zero);
                }
                uint32_t xE2 = 0u;
#pragma unroll
                for (int j = 0; j + 1 < KP; j += 2) xE2 = __vimax3_s16x2(xE2, st[j], st[j + 1]);
                xE2 = __vmaxs2(xE2, st[KP - 1]);
                int xE = max((int)(xE2 & 0xffffu), (int)(xE2 >> 16));
                const bool act = i < L;
                if (act && xE >= limit) ovf = true;
                xE = max(xE - tec, 0);
                xJ = max(xJ, xE);
                xB = max(max(base, xJ) - tjbm, 0);
                if (i == L - 1) resJ = xJ;
            }
            if (__all_sync(0xffffffffu, ovf || (wi * 8 + 8 >= L))) break;
        }
        if (valid) {
            bool pass = true;
            if (!ovf) {
                float sc = ((float)(resJ - tjb) - (float)base);
                sc /= ps.scale_b;
                sc -= 3.0f;
                float seq_score = (float)((double)(sc - nullsc) / kLn2);
                pass = gumbel_surv((double)seq_score, (double)ps.ev[EV_MMU], (double)ps.ev[EV_MLAMBDA]) <= F1;
            }
            if (L == 0) pass = false;       // hmmsearch skips zero-length targets (p7_Pipeline)
            const size_t o = (size_t)(p0 + pl) * ns + sl;
            res[o]  = ovf ? 255 : (uint8_t)resJ;
            flag[o] = pass ? 1 : 0;
        }
    }
}

__global__ void iota_kernel(int32_t *out, int32_t first, int64_t n)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = first + (int32_t)i;
}

// lower_bound of p*ns in the sorted pair list, p = 0..P
__global__ void bounds_kernel(const int32_t *__restrict__ list, const int32_t *__restrict__ n_ptr, int ns, int P,
                              int32_t *__restrict__ bounds)
{
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p > P) return;
    const int n = *n_ptr;
    const long long key = (long long)p * ns;
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if ((long long)list[mid] < key) lo = mid + 1; else hi = mid;
    }
    bounds[p] = lo;
}

// ------------------------------------------------------------------------------------------------
// K5: bias filter -- 2-state HMM Forward with per-row rescaling (Easel esl_hmm_Forward semantics)
__global__ void __launch_bounds__(128)
bias_kernel(const int32_t *__restrict__ list, const int32_t *__restrict__ n_ptr, const int32_t *__restrict__ order,
            int64_t s0, int ns,
            const uint32_t *__restrict__ seqw, const int64_t *__restrict__ woff, const int32_t *__restrict__ seqlen,
            const ProfScalars *__restrict__ pscal, const uint8_t *__restrict__ res,
            const uint8_t *__restrict__ tjbtab, double F1, double F2, float *__restrict__ filtersc, uint8_t *__restrict__ flag2,
            unsigned long long *__restrict__ counters)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= *n_ptr) return;
    const int idx = list[e];
    const int p = idx / ns, sl = idx - p * ns;
    const int64_t s = order[s0 + sl];
    const int L = seqlen[s];
    const uint32_t *w = seqw + woff[s];
    const ProfScalars &ps = pscal[p];
    const float L0 = 400.0f, L1 = (float)ps.M / 8.0f;
    const float t00 = L0 / (L0 + 1.0f), t01 = 1.0f / (L0 + 1.0f);
    const float t10 = 1.0f / (L1 + 1.0f), t11 = L1 / (L1 + 1.0f);
    float logsc = 0.f, mx, d0, d1;
    uint32_t x = residue_at(w, 0);
    d0 = ps.eo[x][0] * 0.999f;
    d1 = ps.eo[x][1] * 0.001f;
    mx = 0.f;
    if (d0 > mx) mx = d0;
    if (d1 > mx) mx = d1;
    d0 /= mx; d1 /= mx;
    logsc += logf_via_double(mx);
    for (int i = 1; i < L; i++) {
        x = residue_at(w, i);
        float n0 = 0.f, n1 = 0.f;
        n0 += d0 * t00; n0 += d1 * t10;
        n1 += d0 * t01; n1 += d1 * t11;
        n0 *= ps.eo[x][0];
        n1 *= ps.eo[x][1];
        mx = 0.f;
        if (n0 > mx) mx = n0;
        if (n1 > mx) mx = n1;
        d0 = n0 / mx; d1 = n1 / mx;
        logsc += logf_via_double(mx);
    }
    float end = 0.f;
    end += d0 * 1.0f;
    end += d1 * 1.0f;
    logsc += logf_via_double(end);
    const float p1 = (float)L / (float)(L + 1);
    const float fsc = logsc + (float)L * logf_via_double(p1) + logf_via_double(1.f - p1);
    filtersc[e] = fsc;
    bool pass = true;
    double Pbias = 0.0;                 // an overflowed MSV score is +inf: P = 0
    const int r = res[(size_t)p * ns + sl];
    if (r != 255) {
        const int tjb = tjbtab[L];
        float sc = ((float)(r - tjb) - (float)ps.base);
        sc /= ps.scale_b;
        sc -= 3.0f;
        float seq_score = (float)((double)(sc - fsc) / kLn2);
        Pbias = gumbel_surv((double)seq_score, (double)ps.ev[EV_MMU], (double)ps.ev[EV_MLAMBDA]);
        pass = Pbias <= F1;
    }
    flag2[e] = pass ? (Pbias > F2 ? 2 : 1) : 0;      // 2: p7_Pipeline would run the Viterbi filter on it (P > F2)
    if (L > 0) atomicAdd(&counters[CNT_BIAS_ROWS], (unsigned long long)L);
}

// ------------------------------------------------------------------------------------------------
// K6: Viterbi filter (HMMER impl_*/vitfilter.c, restated in oracle/ora_hmm.c:viterbi_filter): 16-bit scores in
// 1/500-bit units around base 12000, saturating adds (-32768 = -inf), N / C / J loops free with a -3 nat correction,
// overflow (a match cell at 32767) counts as a pass.  p7_Pipeline runs it only for  F2 < P(MSV + bias) <= F1, which the
// reference's --F1 1e-6 --F2 1e-6 never allows (SeqSample.py:191-209); it is here so that the library is the whole
// hmmsearch cascade under any thresholds (HMMER's own defaults are 0.02 / 1e-3 / 1e-5).  Thread per worklist entry of
// the launch's profile, the row in registers like fb_kernel; max-plus in integers, so any evaluation order is bit-exact:
// M and I descend in place, the D chain ascends.  add-with-floor = one VIADDMNMX; the upper clamp only matters where the
// emission is added, and a row whose best match cell reaches 32767 ends the sequence.
struct VitArgs {
    const int32_t *list;      // the chunk's pair list (all profiles)
    const float   *filtersc;
    const int32_t *vidx;      // this profile's entries that need the filter (P(bias) > F2): indices into list
    int            count;
    const int32_t *order;
    int64_t        s0;
    int            ns, prof;
    const uint32_t *seqw;
    const int64_t  *woff;
    const int32_t  *seqlen;
    const int32_t  *vtab;     // this profile: [MAXM + 2][8] transition words, then [16][48] emission words
    const int16_t  *xwmove;   // per target length
    int             xw_E;
    float           vmu, vlambda;
    double          F2;
    uint8_t        *pass;     // out, per entry
    unsigned long long *counters;
};
constexpr int VIT_T = 0, VIT_E = (MAXM + 2) * 8, VIT_WORDS = (MAXM + 2) * 8 + 16 * 48;
enum { VT_BM = 0, VT_MM, VT_IM, VT_DM, VT_MD, VT_DD, VT_MI, VT_II };

__global__ void __launch_bounds__(128, 3) vit_kernel(const VitArgs a)
{
    __shared__ __align__(16) int32_t s_v[VIT_WORDS];
    for (int t = threadIdx.x; t < VIT_WORDS; t += blockDim.x) s_v[t] = a.vtab[t];
    __syncthreads();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.count) return;
    const int e = a.vidx[j];
    const int idx = a.list[e];
    const int sl = idx - a.prof * a.ns;
    const int64_t s = a.order[a.s0 + sl];
    const int L = a.seqlen[s];
    const uint32_t *w = a.seqw + a.woff[s];
    constexpr int NEG = -32768;
    int Mv[MAXM + 1], Iv[MAXM + 1], Dv[MAXM + 1];
#pragma unroll
    for (int k = 0; k <= MAXM; k++) Mv[k] = Iv[k] = Dv[k] = NEG;
    const int xw_move = a.xwmove[L];
    int xN = 12000, xB = xN + xw_move, xJ = NEG, xC = NEG;
    bool ovf = false;
    for (int i = 1; i <= L && !ovf; i++) {
        const int32_t *em = s_v + VIT_E + residue_at(w, i - 1) * 48;
        int xE = NEG;
        // (the tables are loop-invariant shared-memory reads: without this fence the compiler hoists all 368 of them
        // out of the row loop and spills them)
        asm volatile("" ::: "memory");
#pragma unroll
        for (int k = MAXM; k >= 1; k--) {
            const int4 ta = *(const int4 *)(s_v + VIT_T + (k - 1) * 8), tb = *(const int4 *)(s_v + VIT_T + (k - 1) * 8 + 4);
            const int4 ua = *(const int4 *)(s_v + VIT_T + k * 8), ub = *(const int4 *)(s_v + VIT_T + k * 8 + 4);
            // slots: a = (BM, MM, IM, DM), b = (MD, DD, MI, II)
            int sv = __viaddmax_s32(xB, ua.x, NEG);
            sv = max(sv, __viaddmax_s32(Mv[k - 1], ta.y, NEG));
            sv = max(sv, __viaddmax_s32(Iv[k - 1], ta.z, NEG));
            sv = max(sv, __viaddmax_s32(Dv[k - 1], ta.w, NEG));
            sv = __viaddmax_s32(sv, em[k], NEG);
            const int iv = max(__viaddmax_s32(Mv[k], ub.z, NEG), __viaddmax_s32(Iv[k], ub.w, NEG));
            Mv[k] = sv; Iv[k] = iv;
            xE = max(xE, sv);
            (void)tb;
        }
        int dcur = NEG;
#pragma unroll
        for (int k = 1; k <= MAXM; k++) {
            const int4 tb = *(const int4 *)(s_v + VIT_T + (k - 1) * 8 + 4);
            dcur = max(__viaddmax_s32(Mv[k - 1], tb.x, NEG), __viaddmax_s32(dcur, tb.y, NEG));
            Dv[k] = dcur;
        }
        if (xE >= 32767) { ovf = true; break; }
        xC = max(xC, xE + a.xw_E);
        xJ = max(xJ, xE + a.xw_E);
        xB = max(xJ + xw_move, xN + xw_move);
    }
    bool pass = true;
    if (!ovf) {
        pass = false;
        if (xC > NEG) {
            const float scale_w = 500.0f / (float)kLn2;
            const float sc = ((float)xC + (float)xw_move - 12000.0f) / scale_w - 3.0f;
            const float seq_score = (float)((double)(sc - a.filtersc[e]) / kLn2);
            pass = gumbel_surv((double)seq_score, (double)a.vmu, (double)a.vlambda) <= a.F2;
        }
    }
    a.pass[e] = pass ? 1 : 0;
    atomicAdd(&a.counters[CNT_VIT_ROWS], (unsigned long long)L);
    atomicAdd(&a.counters[CNT_VIT_RUN], 1ull);
}

__global__ void vneed_flag_kernel(const uint8_t *__restrict__ need, int n, uint8_t *__restrict__ run, uint8_t *__restrict__ pass)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    run[e] = need[e] == 2;
    pass[e] = 1;                       // entries the filter does not look at pass
}
// lower_bound of p * ns among the pairs list[vidx[.]] (vidx ascending, list sorted by profile), p = 0..P
__global__ void vbounds_kernel(const int32_t *__restrict__ list, const int32_t *__restrict__ vidx,
                               const int32_t *__restrict__ n_ptr, int ns, int P, int32_t *__restrict__ bounds)
{
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p > P) return;
    const int n = *n_ptr;
    const long long key = (long long)p * ns;
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if ((long long)list[vidx[mid]] < key) lo = mid + 1; else hi = mid;
    }
    bounds[p] = lo;
}

// ------------------------------------------------------------------------------------------------
// K7-K9: Forward -> F3 -> Backward -> domain decoding -> regions.  One warp = one tile of 32 worklist
// entries of the launch's profile; a warp walks tiles persistently and reuses its scratch slab
// spec[row][5][lane] (coalesced 128-byte rows).
struct FbArgs {
    const int32_t *list;      // worklist (pair index = p*ns + sl), this profile's slice
    const float   *filtersc;
    int            count;
    const int32_t *order;     // sequences of the shard sorted by length; s0 indexes into it
    int64_t        s0;
    int            ns, prof;
    const uint32_t *seqw;
    const int64_t  *woff;
    const int32_t  *seqlen;
    const float    *etab;     // [46][16] match odds of this profile
    float          *spec;     // scratch: warps_total * (Lmax+1) * 5 * 32 floats
    int             Lmax;
    float           tau, lambda;
    float           e_move;   // expf(-ln 2) as the host libm rounds it (E->C and E->J, multihit)
    double          F3;
    float          *fwdsc;    // out, per entry
    float          *bcksc;
    uint8_t        *ndom;     // out: number of envelopes (0 if the entry failed F3)
    float          *scale;    // split decode: 1 / bN of every entry that passed F3 (fbdec_kernel's scaleproduct)
    int32_t        *env;      // out: [entry][MAXDOM][2], jenv carries the multidomain flag in bit 30
    unsigned long long *counters;
};

__device__ __forceinline__ void spec_decode(float eraw, float &E, float &S)
{
    if (eraw > 1.0e4f) { E = 1.0f; S = eraw; } else { E = eraw; S = 1.0f; }
}

// ---- TMA (bulk async copy) + mbarrier helpers: a warp streams its own scratch rows back into shared memory ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void tma_row_load(uint32_t dst_smem, const void *src_gmem, uint32_t bytes, uint32_t bar)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst_smem), "l"(src_gmem), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "MBAR_WAIT:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                 "@p bra MBAR_DONE;\n"
                 "bra MBAR_WAIT;\n"
                 "MBAR_DONE:\n"
                 "}" ::"r"(bar), "r"(parity) : "memory");
}

#ifndef FB_DECODE_PF
#define FB_DECODE_PF 16
#endif
__device__ __forceinline__ void l1_prefetch(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

__global__ void __launch_bounds__(FB_THREADS, FB_CTAS_PER_SM)
fb_kernel(const __grid_constant__ ProfConst pc, const FbArgs a)
{
    __shared__ __align__(16) float s_e[16 * ESTRIDE];     // [residue code][node]: odds of the launch's profile
    for (int t = threadIdx.x; t < 16 * ESTRIDE; t += FB_THREADS) {
        const int x = t / ESTRIDE, k = t - x * ESTRIDE;
        s_e[t] = k <= MAXM ? a.etab[k * 16 + x] : 0.f;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int warp_in_grid = (blockIdx.x * FB_THREADS + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * FB_THREADS) >> 5;
    const int ntiles = (a.count + 31) >> 5;
#define SPEC(row, c) sp[((size_t)(row) * SPEC_C + (c)) * 32]

    for (int tile = warp_in_grid; tile < ntiles; tile += nwarps) {
        // the slab of the launch holds every tile: fbdec_kernel reads the rows back
        float *sp = a.spec + (size_t)tile * (size_t)(a.Lmax + 1) * SPEC_C * 32 + lane;
        const int ent = tile * 32 + lane;
        const bool valid = ent < a.count;
        int L = 0;
        const uint32_t *w = a.seqw;
        float filtersc = 0.f;
        if (valid) {
            const int idx = a.list[ent];
            const int sl = idx - a.prof * a.ns;
            const int64_t s = a.order[a.s0 + sl];
            L = a.seqlen[s];
            w = a.seqw + a.woff[s];
            filtersc = a.filtersc[ent];
        }
        int Lw = L;
#pragma unroll
        for (int o = 16; o; o >>= 1) Lw = max(Lw, __shfl_xor_sync(0xffffffffu, Lw, o));

        // length model, multihit (nj = 1)
        const float pmove = (2.0f + 1.0f) / ((float)L + 2.0f + 1.0f);
        const float N_move = pmove, N_loop = 1.0f - pmove;
        const float E_move = a.e_move, E_loop = a.e_move;

        float Mx[MAXM + 2], Ix[MAXM + 2], Dx[MAXM + 2];
#pragma unroll
        for (int k = 0; k <= MAXM + 1; k++) Mx[k] = Ix[k] = Dx[k] = 0.f;

        // ------------------------------ Forward ------------------------------
        float xN = 1.f, xJ = 0.f, xC = 0.f, xE = 0.f, xB = N_move, totscale = 0.f;
        if (valid) { SPEC(0, 0) = 0.f; SPEC(0, 1) = 1.f; SPEC(0, 2) = 0.f; SPEC(0, 3) = xB; SPEC(0, 4) = 0.f; }
        // the residue word (8 nibbles) of rows i..i+7 is fetched one word ahead of its use
        int widx = 0;
        uint32_t wcur = L > 0 ? w[0] : 0u, wnxt = L > 8 ? w[1] : 0u;
        for (int i = 1; i <= Lw; i++) {
            if (((i - 1) >> 3) != widx) {
                widx = (i - 1) >> 3;
                wcur = wnxt;
                wnxt = ((widx + 1) * 8 < L) ? w[widx + 1] : 0u;
            }
            if (i <= L) {
                const float4 *er = (const float4 *)(s_e + ((wcur >> (((i - 1) & 7) * 4)) & 15u) * ESTRIDE);
                // pass 1, descending k, in place: M and I of row i from row i-1 (no serial dependence, so the
                // scheduler needs no far-ahead coefficient loads); pass 2, ascending: the D chain and the E sums.
                // Same operations and summation order as the oracle's single ascending loop.
#pragma unroll
                for (int k = MAXM; k >= 1; k--) {
                    float sv = xB * pc.fa[k][0];
                    sv = fmaf(Mx[k - 1], pc.fa[k][1], sv);
                    sv = fmaf(Ix[k - 1], pc.fa[k][2], sv);
                    sv = fmaf(Dx[k - 1], pc.fa[k][3], sv);
                    sv = sv * EMIS(er, k);
                    const float ic = fmaf(Ix[k], pc.fi[k][0], Mx[k] * pc.fi[k][1]);
                    Mx[k] = sv; Ix[k] = ic;
                }
                float xEm = 0.f, xEd = 0.f, dcur = 0.f;
#pragma unroll
                for (int k = 1; k <= MAXM; k++) {
                    const float dc = fmaf(dcur, pc.fd[k][0], Mx[k - 1] * pc.fd[k][1]);
                    Dx[k] = dc; dcur = dc;
                    xEm += Mx[k]; xEd += dc;
                }
                xE = xEm + xEd;
                xN = xN * N_loop;
                xC = fmaf(xC, N_loop, xE * E_move);
                xJ = fmaf(xJ, N_loop, xE * E_loop);
                xB = fmaf(xJ, N_move, xN * N_move);
                const float eraw = xE;
                if (xE > 1.0e4f) {
                    xN = xN / xE; xC = xC / xE; xJ = xJ / xE; xB = xB / xE;
                    const float inv = 1.0f / xE;
#pragma unroll
                    for (int k = 1; k <= MAXM; k++) { Mx[k] *= inv; Dx[k] *= inv; Ix[k] *= inv; }
                    totscale += logf_via_double(xE);
                    xE = 1.0f;
                }
                SPEC(i, 0) = eraw; SPEC(i, 1) = xN; SPEC(i, 2) = xJ; SPEC(i, 3) = xB; SPEC(i, 4) = xC;
            }
        }
        bool pass = false;
        float fwdsc = 0.f;
        if (valid) {
            fwdsc = totscale + logf_via_double(xC * N_move);
            const float seq_score = (float)((double)(fwdsc - filtersc) / kLn2);
            pass = exp_surv((double)seq_score, (double)a.tau, (double)a.lambda) <= a.F3;
            a.fwdsc[ent] = fwdsc;
        }
        {
            const unsigned m = __ballot_sync(0xffffffffu, pass);
            int rows = valid ? L : 0;
#pragma unroll
            for (int o = 16; o; o >>= 1) rows += __shfl_xor_sync(0xffffffffu, rows, o);
            if (lane == 0) {
                atomicAdd(&a.counters[CNT_FWD_ROWS], (unsigned long long)rows);
                if (m) atomicAdd(&a.counters[CNT_PAST_FWD], (unsigned long long)__popc(m));
            }
            if (m == 0) {
                if (valid) a.ndom[ent] = 0;
                continue;
            }
        }
        if (!pass) L = 0;   // inactive in the Backward sweep
        Lw = L;
#pragma unroll
        for (int o = 16; o; o >>= 1) Lw = max(Lw, __shfl_xor_sync(0xffffffffu, Lw, o));

        // ------------------------------ Backward ------------------------------
        // forward row i is held in f*_i while row i-1 is loaded; products go back in place:
        //   SPEC(i,0) <- (fB[i-1]*bB[i-1])*fS[i-1]      SPEC(i,1) <- (fE[i]*bE[i])*fS[i]
        //   SPEC(i,2..4) <- (fN|fJ|fC[i-1] * bN|bJ|bC[i]) * loop
        float bJ = 0.f, bB = 0.f, bN = 0.f, bC = N_move, bE = bC * E_move, btotscale = 0.f;
        float fE_i = 0.f, fS_i = 1.f;
        if (pass) {
            Dx[MAXM + 1] = 0.f;
#pragma unroll
            for (int k = MAXM; k >= 1; k--) {
                Dx[k] = fmaf(pc.bd1[k - 1], Dx[k + 1], bE);
                Mx[k] = fmaf(pc.bd2[k - 1], Dx[k + 1], bE);
                Ix[k] = 0.f;
            }
            spec_decode(SPEC(L, 0), fE_i, fS_i);
            if (fS_i > 1.0f) {
                bE = bE / fS_i; bN = bN / fS_i; bC = bC / fS_i; bJ = bJ / fS_i; bB = bB / fS_i;
                const float inv = 1.0f / fS_i;
#pragma unroll
                for (int k = 1; k <= MAXM; k++) { Mx[k] *= inv; Dx[k] *= inv; Ix[k] *= inv; }
            }
            btotscale = logf_via_double(fS_i);
        }
        // forward row i-1 (5 specials) is loaded during iteration i+1, the residue word one word ahead
        float qE = 0.f, qN = 0.f, qJ = 0.f, qB = 0.f, qC = 0.f;
        if (Lw >= 1 && Lw - 1 <= L) {
            qE = SPEC(Lw - 1, 0); qN = SPEC(Lw - 1, 1); qJ = SPEC(Lw - 1, 2); qB = SPEC(Lw - 1, 3); qC = SPEC(Lw - 1, 4);
        }
        int bidx = Lw >= 1 ? (Lw - 1) >> 3 : 0;
        uint32_t bcur = (bidx * 8 < L) ? w[bidx] : 0u, bnxt = (bidx >= 1 && (bidx - 1) * 8 < L) ? w[bidx - 1] : 0u;
        for (int i = Lw; i >= 1; i--) {
            const float cE = qE, cN = qN, cJ = qJ, cB = qB, cC = qC;
            if (i >= 2 && i - 2 <= L) {
                qE = SPEC(i - 2, 0); qN = SPEC(i - 2, 1); qJ = SPEC(i - 2, 2); qB = SPEC(i - 2, 3); qC = SPEC(i - 2, 4);
            }
            if (((i - 1) >> 3) != bidx) {
                bidx = (i - 1) >> 3;
                bcur = bnxt;
                bnxt = (bidx >= 1 && (bidx - 1) * 8 < L) ? w[bidx - 1] : 0u;
            }
            if (i <= L) {
                // forward row i-1
                const float fN_p = cN, fJ_p = cJ, fB_p = cB, fC_p = cC;
                float fE_p, fS_p;
                spec_decode(cE, fE_p, fS_p);
                // products that involve backward row i
                SPEC(i, 1) = (fE_i * bE) * fS_i;
                SPEC(i, 2) = (fN_p * bN) * N_loop;
                SPEC(i, 3) = (fJ_p * bJ) * N_loop;
                SPEC(i, 4) = (fC_p * bC) * N_loop;
                if (i > 1) {
                    const float4 *er = (const float4 *)(s_e + ((bcur >> (((i - 1) & 7) * 4)) & 15u) * ESTRIDE);   // x_i
                    bB = 0.f;
#pragma unroll
                    for (int k = 1; k <= MAXM; k++) {
                        Mx[k] = Mx[k] * EMIS(er, k);
                        bB = fmaf(Mx[k], pc.bm[k - 1], bB);
                    }
                    bC = bC * N_loop;
                    bJ = fmaf(bB, N_move, bJ * N_loop);
                    bN = fmaf(bB, N_move, bN * N_loop);
                    bE = fmaf(bC, E_move, bJ * E_loop);
                    Dx[MAXM + 1] = 0.f;
                    float mnext = 0.f;
#pragma unroll
                    for (int k = MAXM; k >= 1; k--) {
                        const float mpe_k = Mx[k];
                        const float ic = fmaf(mnext, pc.ba[k][0], Ix[k] * pc.ba[k][1]);
                        // every M and D state also exits to E: bE is the addend the FMA chains start from
                        const float dc = fmaf(mnext, pc.bd0[k - 1], fmaf(Dx[k + 1], pc.bd1[k - 1], bE));
                        const float mc = fmaf(mnext, pc.ba[k][2], fmaf(Ix[k], pc.ba[k][3], fmaf(Dx[k + 1], pc.bd2[k - 1], bE)));
                        Mx[k] = mc; Ix[k] = ic; Dx[k] = dc;
                        mnext = mpe_k;
                    }
                    if (fS_p > 1.0f) {
                        bE = bE / fS_p; bN = bN / fS_p; bC = bC / fS_p; bJ = bJ / fS_p; bB = bB / fS_p;
                        const float inv = 1.0f / fS_p;
#pragma unroll
                        for (int k = 1; k <= MAXM; k++) { Mx[k] *= inv; Dx[k] *= inv; Ix[k] *= inv; }
                        btotscale += logf_via_double(fS_p);     // log(1) == +0 exactly: rows without a rescale add nothing
                    }
                } else {
                    // row 0: only B and N are live
                    const float4 *er = (const float4 *)(s_e + (bcur & 15u) * ESTRIDE);
                    bB = 0.f;
#pragma unroll
                    for (int k = 1; k <= MAXM; k++) bB = fmaf(Mx[k] * EMIS(er, k), pc.bm[k - 1], bB);
                    bN = fmaf(bB, N_move, bN * N_loop);
                }
                SPEC(i, 0) = (fB_p * bB) * fS_p;
                fE_i = fE_p; fS_i = fS_p;
            }
        }

        if (pass) {
            a.bcksc[ent] = btotscale + logf_via_double(bN);
            a.scale[ent] = 1.0f / bN;
        }
        if (valid) a.ndom[ent] = pass ? 1 : 0;      // fbdec_kernel replaces the mark by the number of envelopes
    }
#undef SPEC
}

// K9a: posterior decoding + region finding of every entry that passed F3: one lane per entry over the launch's slab
// ([tile][row][5][lane], coalesced 128-byte rows), light on registers so that many warps hide the row-to-row latency
__global__ void __launch_bounds__(128) fbdec_kernel(const FbArgs a)
{
    const int lane = threadIdx.x & 31;
    const int tile = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int ent = tile * 32 + lane;
    if (ent >= a.count || a.ndom[ent] == 0) return;
    const int idx = a.list[ent];
    const int sl = idx - a.prof * a.ns;
    const int64_t sq = a.order[a.s0 + sl];
    const int L = a.seqlen[sq];
    float *sp = a.spec + (size_t)tile * (size_t)(a.Lmax + 1) * SPEC_C * 32 + lane;
#define SPEC(row, c) sp[((size_t)(row) * SPEC_C + (c)) * 32]
    int nd = 0;
    {
    const float scaleproduct = a.scale[ent];
    const float rt1 = 0.25f, rt2 = 0.10f, rt3 = 0.20f;
    float btot = 0.f, etot = 0.f;
    int ri = -1;
    bool triggered = false;
    int nmulti = 0;
    SPEC(0, 0) = 0.f; SPEC(0, 1) = 0.f;   // btot[0], etot[0]
#if FB_DECODE_PF > 0
    // rows FB_DECODE_PF ahead are pulled into L1 (CCTL.PF1: no register, no unrolling); the row-ahead register
    // loads below then hit L1 instead of waiting out an HBM round trip per row
#pragma unroll 1
    for (int j = 2; j <= FB_DECODE_PF && j <= L; j++) {
#pragma unroll
        for (int cc = 0; cc < SPEC_C; cc++) l1_prefetch(&SPEC(j, cc));
    }
#endif
    float r0 = SPEC(1, 0), r1 = SPEC(1, 1), r2 = SPEC(1, 2), r3 = SPEC(1, 3), r4 = SPEC(1, 4);
    for (int j = 1; j <= L; j++) {
#if FB_DECODE_PF > 0
        if (j + FB_DECODE_PF <= L) {
#pragma unroll
            for (int cc = 0; cc < SPEC_C; cc++) l1_prefetch(&SPEC(j + FB_DECODE_PF, cc));
        }
#endif
        const float v0 = r0, v1 = r1, v2 = r2, v3 = r3, v4 = r4;
        if (j < L) { r0 = SPEC(j + 1, 0); r1 = SPEC(j + 1, 1); r2 = SPEC(j + 1, 2); r3 = SPEC(j + 1, 3); r4 = SPEC(j + 1, 4); }
        const float db = v0 * scaleproduct, de = v1 * scaleproduct;
        const float btot_p = btot, etot_p = etot;
        btot = btot + db;
        etot = etot + de;
        float njcp = v2 * scaleproduct;
        njcp += v3 * scaleproduct;
        njcp += v4 * scaleproduct;
        const float mocc = 1.f - njcp;
        SPEC(j, 0) = btot; SPEC(j, 1) = etot;
        if (!triggered) {
            if (mocc - (btot - btot_p) < rt2) ri = j;
            else if (ri == -1) ri = j;
            if (mocc >= rt1) triggered = true;
        } else if (mocc - (etot - etot_p) < rt2) {
            float mx = -1.0f;
            const float e0 = SPEC(ri - 1, 1);
            for (int z = ri; z <= j; z++) {
                const float x1 = SPEC(z, 1) - e0, x2 = btot - SPEC(z - 1, 0);
                const float en = x1 < x2 ? x1 : x2;
                if (en > mx) mx = en;
            }
            const int multi = mx >= rt3;
            nmulti += multi;
            if (nd < ITSX_MAXDOM) {
                a.env[((size_t)ent * ITSX_MAXDOM + nd) * 2 + 0] = ri;
                a.env[((size_t)ent * ITSX_MAXDOM + nd) * 2 + 1] = j | (multi << 30);
                nd++;
            } else {
                atomicAdd(&a.counters[CNT_DOM_OVERFLOW], 1ull);
            }
            ri = -1;
            triggered = false;
        }
    }
    if (nmulti) atomicAdd(&a.counters[CNT_MULTI], (unsigned long long)nmulti);
    atomicAdd(&a.counters[CNT_BCK_ROWS], (unsigned long long)L);
    }
    a.ndom[ent] = (uint8_t)nd;
#undef SPEC
}

// ------------------------------------------------------------------------------------------------
// K9b: multidomain regions (p7_domaindef.c: region_trace_ensemble + p7_spensemble_Cluster; SURVEY A.5), operation
// for operation the same as oracle/ora_hmm.c:resolve_multidomain.  About 1 % of the regions, but 200 stochastic
// tracebacks each, so the stage is split so that the TRACE is the unit of parallelism:
//   mdfwd_kernel    one thread per region: multihit Forward over the region, full (M, I, D) matrix and the per-row
//                   normalised C / J / B choices to a region-private slab in HBM
//   mdtrace_kernel  one thread per (region, trace): the random walk back through the matrix with HMMER's "fast"
//                   generator leap-frogged to substream t (x_(t 2^20)); the 200 lanes of a region read the same slab
//                   (L1 / L2 resident); phases of the walk are warp-vote loops so lanes stay converged; a trace
//                   leaves its domains (coordinates + null2 odds by trace) in a fixed 100-byte record
//   mdclust_kernel  one warp per region: n2sc per position, distinct segments, single-linkage clustering,
//                   cluster envelopes (start order) with their domcorrection
//   mdapply_kernel  one thread per worklist entry: the cluster envelopes replace the region in the entry's list.
// The cluster envelopes carry bit 29 ("null2 done"): env_kernel still gives their unihit Forward score, final_kernel
// takes their domcorrection from envdc[] and the region-wide sum of the trace n2sc from n2reg[].
constexpr int MD_NSAMPLES = 200;
constexpr int MD_MAXTDOM = 4;                  // domains kept per trace
constexpr int MD_W = MAXM + 1;
constexpr int MD_STREAM_LOG2 = 20;
struct MdRow { float pC0, pC1, pJ0, pJ1, pB0, pB1, nrmE, xB; };   // per row: normalised C / J / B choices, 1 / xE, xB
struct MdDom { uint16_t from, to; uint8_t k, m; uint16_t pad; float n2[4]; };   // region-relative rows
struct MdTrace { int32_t nd; MdDom d[MD_MAXTDOM]; };                             // a trace while it is walked (registers)
// The traces of a region in HBM, arrays over the trace index so that 32 traces are written and read with coalesced
// accesses: nd[200] | from, to [4][200] | k, m [4][200] | null2 odds [4][200] float4
constexpr int MD_TRACE_FT = MD_NSAMPLES * 4;
constexpr int MD_TRACE_KM = MD_TRACE_FT + MD_MAXTDOM * MD_NSAMPLES * 4;
constexpr int MD_TRACE_N2 = MD_TRACE_KM + MD_MAXTDOM * MD_NSAMPLES * 4;
constexpr int MD_TRACE_BYTES = MD_TRACE_N2 + MD_MAXTDOM * MD_NSAMPLES * 16;
static_assert(MD_TRACE_N2 % 16 == 0 && MD_TRACE_BYTES % 16 == 0, "float4 alignment of the trace arrays");
struct MdRes { int32_t n; float regsum; int32_t ci[ITSX_MAXDOM], cj[ITSX_MAXDOM]; float cdc[ITSX_MAXDOM]; };
struct MdArgs {
    // regions of this chunk: [r0, r1) of the region list
    int             r0, r1;
    const int32_t  *reg_ent;  // worklist entry of every region
    const int32_t  *reg_i, *reg_j;
    const int32_t  *reg_row;  // first row of the region's slab (prefix sum of Ld + 1), relative to the list
    int             row0;     // reg_row of region r0
    const int32_t *list;
    const int32_t *order;
    int64_t        s0;
    int            ns;
    const uint32_t *seqw;
    const int64_t  *woff;
    const int32_t  *seqlen;
    const float    *mdtab;    // [P][MAXM + 2][8]: transitions out of node k, B->M_k in slot 7
    const float    *etab;     // [P][MAXM + 1][16]
    const ProfScalars *pscal;
    float4         *cell;     // [row][MD_W]: (M, I, D, -)
    MdRow          *rowrec;   // [row]
    char           *trace;    // [region - r0][MD_TRACE_BYTES]
    MdRes          *res;      // [region]
    char           *scratch;  // mdclust: per thread
    size_t          per_thread;
    int             maxrows;
    float           e_move;
    unsigned long long *counters;
};
struct MdStreams { uint32_t x[MD_NSAMPLES]; };
__device__ __forceinline__ double md_rng(uint32_t &x)
{
    x = x * 69069u + 1u;
    return (double)x / 4294967296.0;
}
// esl_vec_FNorm
__device__ __forceinline__ void md_norm(float *p, int n)
{
    float sum = 0.f;
    for (int a = 0; a < n; a++) sum += p[a];
    if (sum != 0.f) { const float inv = 1.0f / sum; for (int a = 0; a < n; a++) p[a] = p[a] * inv; }   // esl_vec_FScale(1/sum)
    else { for (int a = 0; a < n; a++) p[a] = 1.0f / (float)n; }
}
__device__ __forceinline__ int md_pick2(uint32_t &rng, float p0, float p1)
{
    for (;;) {
        const double roll = md_rng(rng);
        float c = 0.f;
        c += p0; if (roll < (double)c) return 0;
        c += p1; if (roll < (double)c) return 1;
    }
}
enum { MS_M = 0, MS_D, MS_I, MS_N, MS_C, MS_J, MS_E, MS_B, MS_S };

struct MdRegion { int L, M, ireg, Ld; const uint32_t *w; const float *tp, *et; };
__device__ __forceinline__ MdRegion md_region(const MdArgs &a, int r)
{
    MdRegion g;
    const int e = a.reg_ent[r];
    const int idx = a.list[e];
    const int p = idx / a.ns, sl = idx - p * a.ns;
    const int64_t s = a.order[a.s0 + sl];
    g.L = a.seqlen[s];
    g.w = a.seqw + a.woff[s];
    g.M = a.pscal[p].M;
    g.tp = a.mdtab + (size_t)p * (MAXM + 2) * 8;
    g.et = a.etab + (size_t)p * (MAXM + 1) * 16;
    g.ireg = a.reg_i[r];
    g.Ld = a.reg_j[r] - g.ireg + 1;
    return g;
}

// ---- multihit Forward over the region, full matrix (oracle forward_engine), and the per-row choice tables ----
__global__ void __launch_bounds__(64) mdfwd_kernel(const MdArgs a)
{
    constexpr unsigned FULL = 0xffffffffu;
    const int r = a.r0 + blockIdx.x * blockDim.x + threadIdx.x;
    const bool act = r < a.r1;
    MdRegion g;
    g.L = 1; g.M = 1; g.ireg = 1; g.Ld = 0; g.w = a.seqw; g.tp = a.mdtab; g.et = a.etab;
    size_t row0 = 0;
    if (act) { g = md_region(a, r); row0 = (size_t)(a.reg_row[r] - a.row0); }
    float4 *cell = a.cell + row0 * MD_W;
    MdRow *rowrec = a.rowrec + row0;
    const int M = g.M, Ld = g.Ld;
    const float *tp = g.tp, *et = g.et;
#define CELL(i, k) cell[(size_t)(i) * MD_W + (k)]
    const float pmove = (2.0f + 1.0f) / ((float)g.L + 2.0f + 1.0f);
    const float N_move = pmove, N_loop = 1.0f - pmove, E_move = a.e_move, E_loop = a.e_move;
    float xN = 1.f, xJ = 0.f, xC = 0.f, xE = 0.f, xB = N_move;
    if (act) {
        for (int k = 0; k <= M; k++) CELL(0, k) = make_float4(0.f, 0.f, 0.f, 0.f);
        MdRow r0;
        float pb[2] = {xN * N_move, xJ * N_move};
        md_norm(pb, 2);
        r0.pC0 = r0.pC1 = r0.pJ0 = r0.pJ1 = 0.f; r0.pB0 = pb[0]; r0.pB1 = pb[1]; r0.nrmE = 0.f; r0.xB = xB;
        rowrec[0] = r0;
    }
    int Ldw = Ld;
#pragma unroll
    for (int o = 16; o; o >>= 1) Ldw = max(Ldw, __shfl_xor_sync(FULL, Ldw, o));
    for (int i = 1; i <= Ldw; i++) {
        if (i > Ld) continue;
        const uint32_t x = residue_at(g.w, g.ireg - 1 + i - 1);
        const float cprev = xC, jprev = xJ;          // stored (scaled) specials of row i-1
        float mcur = 0.f, dcur = 0.f, xEm = 0.f, xEd = 0.f;
        CELL(i, 0) = make_float4(0.f, 0.f, 0.f, 0.f);
        float4 pk1 = CELL(i - 1, 0);                 // row i-1, node k-1
        for (int k = 1; k <= M; k++) {
            const float4 pk = CELL(i - 1, k);
            const float4 t1a = __ldg((const float4 *)(tp + (k - 1) * 8)), t1b = __ldg((const float4 *)(tp + (k - 1) * 8 + 4));
            const float4 ta = __ldg((const float4 *)(tp + k * 8)), tb = __ldg((const float4 *)(tp + k * 8 + 4));
            // slots: a = (MM, MI, MD, IM), b = (II, DM, DD, BM)
            float sv = xB * tb.w;
            sv = fmaf(pk1.x, t1a.x, sv);
            sv = fmaf(pk1.y, t1a.w, sv);
            sv = fmaf(pk1.z, t1b.y, sv);
            sv = sv * __ldg(et + k * 16 + x);
            const float dc = fmaf(dcur, t1b.z, mcur * t1a.z);
            const float ic = fmaf(pk.y, tb.x, pk.x * ta.y);
            CELL(i, k) = make_float4(sv, ic, dc, 0.f);
            xEm += sv; xEd += dc;
            mcur = sv; dcur = dc;
            pk1 = pk;
        }
        xE = xEm + xEd;
        xN = xN * N_loop;
        xC = fmaf(xC, N_loop, xE * E_move);
        xJ = fmaf(xJ, N_loop, xE * E_loop);
        xB = fmaf(xJ, N_move, xN * N_move);
        float sc = 1.0f;
        if (xE > 1.0e4f) {
            xN = xN / xE; xC = xC / xE; xJ = xJ / xE; xB = xB / xE;
            const float inv = 1.0f / xE;
            for (int k = 1; k <= M; k++) {
                float4 v = CELL(i, k);
                v.x *= inv; v.z *= inv; v.y *= inv;
                CELL(i, k) = v;
            }
            sc = xE;
            xE = 1.0f;
        }
        MdRow rr;
        float pc[2] = {cprev * N_loop, xE * E_move * sc};
        md_norm(pc, 2);
        float pj[2] = {jprev * N_loop, xE * E_loop * sc};
        md_norm(pj, 2);
        float pb[2] = {xN * N_move, xJ * N_move};
        md_norm(pb, 2);
        rr.pC0 = pc[0]; rr.pC1 = pc[1]; rr.pJ0 = pj[0]; rr.pJ1 = pj[1]; rr.pB0 = pb[0]; rr.pB1 = pb[1];
        rr.nrmE = (float)(1.0 / (double)xE);
        rr.xB = xB;
        rowrec[i] = rr;
    }
#undef CELL
}

// ---- one stochastic traceback per thread.  A trace is  C..C E [domain] B ( N.. | J..J E [domain] B ... ).  The N walk
// draws no random numbers and is skipped.  Every phase is a loop on a warp vote, the domain step is one predicated
// code path for M, D and I. ----
__global__ void __launch_bounds__(128) mdtrace_kernel(const MdArgs a, const __grid_constant__ MdStreams streams)
{
    constexpr unsigned FULL = 0xffffffffu;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int r = a.r0 + (int)(gid / MD_NSAMPLES), t = (int)(gid % MD_NSAMPLES);
    const bool act = r < a.r1;
    MdRegion g;
    g.L = 1; g.M = 1; g.ireg = 1; g.Ld = 0; g.w = a.seqw; g.tp = a.mdtab; g.et = a.etab;
    size_t row0 = 0;
    if (act) { g = md_region(a, r); row0 = (size_t)(a.reg_row[r] - a.row0); }
    const float4 *cell = a.cell + row0 * MD_W;
    const MdRow *rowrec = a.rowrec + row0;
    const int M = g.M;
    const float *tp = g.tp, *et = g.et;
#define CELL(i, k) cell[(size_t)(i) * MD_W + (k)]
    const int Q = max(((M - 1) / 4) + 1, 2);
    uint32_t rng = streams.x[t];
    MdTrace out;
    out.nd = 0;
    int i = g.Ld, k = 0;
    bool inJ = false, alive = act;
    while (__any_sync(FULL, alive)) {
        // ---- C (or J) walk: stay with p0 (i--), leave to E with p1 ----
        bool walking = alive;
        while (__any_sync(FULL, walking)) {
            if (walking) {
                const MdRow &rr = rowrec[i];
                if (md_pick2(rng, inJ ? rr.pJ0 : rr.pC0, inJ ? rr.pJ1 : rr.pC1) != 0 || i <= 1) walking = false;
                else i--;       // (i <= 1 is unreachable: C(0) = J(0) = 0)
            }
        }
        // ---- E at row i: M_k / D_k in striped order, scaled by 1 / xE(i) ----
        int st = MS_B;
        if (alive) {
            const double roll = md_rng(rng);
            const float nrm = rowrec[i].nrmE;
            double sum = 0.0;
            bool done = false;
            st = MS_M;
            while (!done) {
                for (int q = 0; q < Q && !done; q++) {
                    float4 cc[4];
                    for (int rr = 0; rr < 4; rr++) {
                        const int kk = rr * Q + q + 1;
                        cc[rr] = kk <= M ? CELL(i, kk) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                    for (int rr = 0; rr < 4 && !done; rr++) {
                        sum += (double)(cc[rr].x * nrm);
                        if (roll < sum) { k = rr * Q + q + 1; st = MS_M; done = true; }
                    }
                    for (int rr = 0; rr < 4 && !done; rr++) {
                        sum += (double)(cc[rr].z * nrm);
                        if (roll < sum) { k = rr * Q + q + 1; st = MS_D; done = true; }
                    }
                }
                if (!done && sum < 0.99) { k = 1; st = MS_M; done = true; }
            }
        }
        __syncwarp();
        // ---- domain walk back to B; null2 odds are summed in walk order ----
        int d_to = 0, d_m = 0, d_from = 0, d_k = 0, nI = 0;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        while (__any_sync(FULL, st != MS_B)) {
            if (st == MS_B) continue;
            if (st == MS_M) {
                if (d_to == 0) { d_to = i; d_m = k; }
                d_from = i; d_k = k;
                const float4 e4 = __ldg((const float4 *)(et + k * 16));
                s0 += e4.x; s1 += e4.y; s2 += e4.z; s3 += e4.w;
            } else if (st == MS_I) {
                nI++;
            }
            // predecessor of state st at (i, k): one cell, the transitions out of its node
            const int ri = st == MS_D ? i : i - 1, kc = st == MS_I ? k : k - 1;
            const float4 c1 = CELL(ri, kc);
            const float4 ta = __ldg((const float4 *)(tp + kc * 8)), tb = __ldg((const float4 *)(tp + kc * 8 + 4));
            float path[4];
            int n;
            if (st == MS_M) {
                path[0] = rowrec[i - 1].xB * __ldg(tp + k * 8 + 7);
                path[1] = c1.x * ta.x; path[2] = c1.y * ta.w; path[3] = c1.z * tb.y;
                n = 4;
            } else if (st == MS_D) {
                path[0] = c1.x * ta.z; path[1] = c1.z * tb.z; path[2] = 0.f; path[3] = 0.f;
                n = 2;
            } else {
                path[0] = c1.x * ta.y; path[1] = c1.y * tb.x; path[2] = 0.f; path[3] = 0.f;
                n = 2;
            }
            // esl_vec_FNorm over the n live paths (the padded zeros leave the float sums unchanged)
            float sum = 0.f;
            sum += path[0]; sum += path[1]; sum += path[2]; sum += path[3];
            if (sum != 0.f) {
                const float inv = 1.0f / sum;
                path[0] = path[0] * inv; path[1] = path[1] * inv; path[2] = path[2] * inv; path[3] = path[3] * inv;
            } else {
                const float u = 1.0f / (float)n;
                path[0] = u; path[1] = u;
                if (n == 4) { path[2] = u; path[3] = u; }
            }
            int c;
            for (;;) {
                const double roll = md_rng(rng);
                float cs = 0.f;
                cs += path[0]; if (roll < (double)cs) { c = 0; break; }
                cs += path[1]; if (roll < (double)cs) { c = 1; break; }
                if (n == 4) {
                    cs += path[2]; if (roll < (double)cs) { c = 2; break; }
                    cs += path[3]; if (roll < (double)cs) { c = 3; break; }
                }
            }
            if (st == MS_M) { st = c == 0 ? MS_B : c == 1 ? MS_M : c == 2 ? MS_I : MS_D; k--; i--; }
            else if (st == MS_D) { st = c == 0 ? MS_M : MS_D; k--; }
            else { st = c == 0 ? MS_M : MS_I; i--; }
        }
        if (alive) {
            if (out.nd < MD_MAXTDOM) {
                const float norm = 1.0f / (float)(d_to - d_from + 1), fi = (float)nI;
                MdDom &dd = out.d[out.nd];
                dd.from = (uint16_t)d_from; dd.to = (uint16_t)d_to; dd.k = (uint8_t)d_k; dd.m = (uint8_t)d_m; dd.pad = 0;
                dd.n2[0] = (s0 + fi) * norm; dd.n2[1] = (s1 + fi) * norm;
                dd.n2[2] = (s2 + fi) * norm; dd.n2[3] = (s3 + fi) * norm;
                out.nd++;
            }
            // ---- B at row i: N ends the trace, J goes on ----
            const MdRow &rr = rowrec[i];
            if (md_pick2(rng, rr.pB0, rr.pB1) == 0) alive = false;
            inJ = true;
        }
    }
    if (act) {
        char *tb = a.trace + (size_t)(r - a.r0) * MD_TRACE_BYTES;
        ((int32_t *)tb)[t] = out.nd;
        for (int d = 0; d < out.nd; d++) {
            const MdDom &dd = out.d[d];
            ((uint32_t *)(tb + MD_TRACE_FT))[d * MD_NSAMPLES + t] = (uint32_t)dd.from | ((uint32_t)dd.to << 16);
            ((uint32_t *)(tb + MD_TRACE_KM))[d * MD_NSAMPLES + t] = (uint32_t)dd.k | ((uint32_t)dd.m << 8);
            ((float4 *)(tb + MD_TRACE_N2))[d * MD_NSAMPLES + t] = make_float4(dd.n2[0], dd.n2[1], dd.n2[2], dd.n2[3]);
        }
    }
#undef CELL
}

// ---- per region, one WARP: n2sc, distinct segments, single linkage clustering, cluster envelopes.  Every phase is
// lane-parallel and reads the trace records with coalesced loads, one round trip per 32 traces (the first version walked
// the 200 records one after the other: two dependent HBM latencies per trace, 0.43 ms per region).  Only the float sums
// keep the oracle's order (per position: samples in trace order; per envelope and per region: positions ascending).
//   A. 32 traces per round: lanes load their trace's domains (left to right), scan the counts into the flat sample
//      list (key + trace per sample, for B-D) and stage the round's samples in shared memory; then lanes own positions
//      (up to four blocks of 32 per pass over the traces) and sum the null2 odds of the covering samples in registers
//   B. distinct segments through a shared-memory hash table (the slot keeps the FIRST sample with that key, so the
//      segments are numbered in order of first appearance like a serial scan would), multiplicities by atomics
//   C. level-synchronous component search: lanes own unassigned segments and test them against the frontier
//   D. traces per cluster by atomics; envelope end points from a histogram of the cluster's starts / ends
constexpr int MDC_WARPS = 4;
constexpr int MDC_CAP = 832;                   // >= MD_NSAMPLES * MD_MAXTDOM, a multiple of 32
constexpr int MDC_HT = 1024;                   // hash slots (power of two > MDC_CAP); later the end-point histogram
constexpr int MDC_PB = 4;                      // position blocks (of 32) per pass over the traces
static_assert(MDC_CAP >= MD_NSAMPLES * MD_MAXTDOM && MDC_CAP % 32 == 0 && MDC_HT > MDC_CAP, "mdclust capacities");
struct MdClustSmem {
    unsigned long long skey[MDC_CAP];          // distinct segments: i | j << 16 | (i - k) << 32 | (j - m) << 48
    uint32_t htab[MDC_HT];
    uint32_t scount[MDC_CAP];                  // how many samples hit the segment
    int16_t  asg[MDC_CAP];
    int16_t  queue[MDC_CAP];                   // component search: assigned segments in discovery order
};
__host__ __device__ inline size_t md_clust_bytes(int maxrows)
{
    // per warp: sample keys, n2sc per row, sample -> slot / segment, sample -> trace
    size_t b = (size_t)MDC_CAP * 8 + (size_t)(maxrows + 1) * 4 + (size_t)MDC_CAP * (2 + 1);
    return (b + 255) / 256 * 256;
}
// link_spsamples on segments stored as four 16-bit fields  i | j << 16 | (i - k) << 32 | (j - m) << 48  (the two
// diagonals are what most pairs of different domains differ in, so they are tested first; the conjunction is the same).
// (float)nov / (float)n < 0.8f  is decided exactly by  5 nov < 4 n : for n < 2^16 the quotient is either 4/5 (rounds to
// 0.8f, not smaller) or at least 1 / (5 n) > 3e-6 away from it, far more than a float ulp.
__device__ __forceinline__ unsigned long long md_seg_word(unsigned long long key)
{
    const int i = (int)(key & 0xffffu), j = (int)((key >> 16) & 0xffffu), k = (int)((key >> 32) & 0xffu), m = (int)((key >> 40) & 0xffu);
    return (unsigned long long)(uint32_t)(i | (j << 16)) |
           ((unsigned long long)(uint32_t)(((i - k) & 0xffff) | (((j - m) & 0xffff) << 16)) << 32);
}
__device__ __forceinline__ bool md_link_word(unsigned long long wa, unsigned long long wb)
{
    const uint32_t alo = (uint32_t)wa, blo = (uint32_t)wb, ahi = (uint32_t)(wa >> 32), bhi = (uint32_t)(wb >> 32);
    // differences of the 16-bit diagonal fields, modulo 2^16 (exact: positions are below 2^16, nodes below 2^8)
    const int dd = (int)(short)(uint16_t)((ahi & 0xffffu) - (bhi & 0xffffu)), de = (int)(short)(uint16_t)((ahi >> 16) - (bhi >> 16));
    if ((unsigned)(dd + 4) > 8u) return false;
    if ((unsigned)(de + 4) > 8u) return false;
    const int ai = (int)(alo & 0xffffu), aj = (int)(alo >> 16), bi = (int)(blo & 0xffffu), bj = (int)(blo >> 16);
    int nov = min(aj, bj) - max(ai, bi) + 1;
    int n = min(aj - ai + 1, bj - bi + 1);
    if (5 * nov < 4 * n) return false;
    const int ak = (ai - (int)(ahi & 0xffffu)) & 0xffff, am = (aj - (int)(ahi >> 16)) & 0xffff;
    const int bk = (bi - (int)(bhi & 0xffffu)) & 0xffff, bm = (bj - (int)(bhi >> 16)) & 0xffff;
    nov = min(am, bm) - max(ak, bk) + 1;
    n = min(am - ak + 1, bm - bk + 1);
    return 5 * nov >= 4 * n;
}
// null2 odds of an IUPAC residue code x under a domain's (A, C, G, T) odds: the average of its bases in base order; N is 1
__device__ __noinline__ float md_null2_iupac(uint32_t x, float a, float c, float g, float t)
{
    if (x == 15) return 1.0f;
    const uint32_t dmask = (uint32_t)(0x0FD7EB96C3A58421ull >> (4 * x)) & 15u;
    float sa = 0.f;
    int na = 0;
    if (dmask & 1u) { sa += a; na++; }
    if (dmask & 2u) { sa += c; na++; }
    if (dmask & 4u) { sa += g; na++; }
    if (dmask & 8u) { sa += t; na++; }
    return sa / (float)na;
}
// lanes own positions (pos0 + 32 b): the staged samples in order, each adds its odds where it covers the position
template <int NB, bool PLAIN>
__device__ __forceinline__ void md_accumulate(const uint32_t *st_ft, const float4 *st_n2, int count, int pos0,
                                              const uint32_t (&x)[MDC_PB], float (&sum)[MDC_PB], int (&cover)[MDC_PB])
{
    static_assert(NB <= MDC_PB, "position blocks per pass");
#pragma unroll 4
    for (int q = 0; q < count; q++) {
        const uint32_t f = st_ft[q];
        const int from = (int)(f & 0xffffu), len = (int)(f >> 16) - from;
        const float *o = (const float *)(st_n2 + q);
#pragma unroll
        for (int b = 0; b < NB; b++) {
            if ((unsigned)(pos0 + 32 * b - from) <= (unsigned)len) {
                float v;
                if (PLAIN || x[b] < 4u) v = o[x[b] & 3u];
                else v = md_null2_iupac(x[b], o[0], o[1], o[2], o[3]);
                sum[b] += v;
                cover[b]++;
            }
        }
    }
}
template <bool PLAIN>
__device__ __forceinline__ void md_accumulate_nb(int nb, const uint32_t *st_ft, const float4 *st_n2, int count, int pos0,
                                                 const uint32_t (&x)[MDC_PB], float (&sum)[MDC_PB], int (&cover)[MDC_PB])
{
    switch (nb) {
    case 1: md_accumulate<1, PLAIN>(st_ft, st_n2, count, pos0, x, sum, cover); break;
    case 2: md_accumulate<2, PLAIN>(st_ft, st_n2, count, pos0, x, sum, cover); break;
    case 3: md_accumulate<3, PLAIN>(st_ft, st_n2, count, pos0, x, sum, cover); break;
    default: md_accumulate<4, PLAIN>(st_ft, st_n2, count, pos0, x, sum, cover); break;
    }
}
__global__ void __launch_bounds__(MDC_WARPS * 32) mdclust_kernel(const MdArgs a)
{
    constexpr unsigned FULL = 0xffffffffu;
    constexpr uint32_t EMPTY = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char mdc_smem[];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int warp = blockIdx.x * MDC_WARPS + wid, nwarps = gridDim.x * MDC_WARPS;
    const unsigned lt = (1u << lane) - 1u;
    MdClustSmem &sm = ((MdClustSmem *)mdc_smem)[wid];
    char *scr = a.scratch + (size_t)warp * a.per_thread;
    unsigned long long *rkey = (unsigned long long *)scr;            // [MDC_CAP]
    float *acc = (float *)(rkey + MDC_CAP);                          // [maxrows + 1]
    uint16_t *rslot = (uint16_t *)(acc + (a.maxrows + 1));           // [MDC_CAP]: hash slot, then segment id
    uint8_t *rtr = (uint8_t *)(rslot + MDC_CAP);                     // [MDC_CAP]: trace of the sample
    for (int r = a.r0 + warp; r < a.r1; r += nwarps) {
        const MdRegion g = md_region(a, r);
        const int Ld = g.Ld, ireg = g.ireg;
        const char *tb = a.trace + (size_t)(r - a.r0) * MD_TRACE_BYTES;
        const int32_t *t_nd = (const int32_t *)tb;
        const uint32_t *t_ft = (const uint32_t *)(tb + MD_TRACE_FT), *t_km = (const uint32_t *)(tb + MD_TRACE_KM);
        const float4 *t_n2 = (const float4 *)(tb + MD_TRACE_N2);
        // ---- A. flat sample list + n2sc per position ----
        // the samples of one round (32 traces, left to right within a trace) are staged in the segment area, which
        // phase B only fills afterwards: from | to << 16 and the four null2 odds per sample
        uint32_t *st_ft = (uint32_t *)sm.skey;                       // [32 * MD_MAXTDOM]
        float4 *st_n2 = (float4 *)(sm.skey + 16 * MD_MAXTDOM);       // [32 * MD_MAXTDOM]
        int nraw = 0;
        for (int pg = 1; pg <= Ld; pg += 32 * MDC_PB) {
            const bool first_pass = pg == 1;
            const int nb = min(MDC_PB, (Ld - pg + 32) >> 5);         // position blocks of this pass
            uint32_t x[MDC_PB];
            float sum[MDC_PB];
            int cover[MDC_PB];
            bool plain = true;                     // no IUPAC / N residue among this pass's positions (warp-uniform)
#pragma unroll
            for (int b = 0; b < MDC_PB; b++) {
                const int pos = pg + 32 * b + lane;
                x[b] = pos <= Ld ? residue_at(g.w, ireg - 1 + pos - 1) : 0u;
                sum[b] = 0.f; cover[b] = 0;
                plain = plain && !__any_sync(FULL, x[b] >= 4u);
            }
            for (int t0 = 0; t0 < MD_NSAMPLES; t0 += 32) {
                const int t = t0 + lane, tt = min(t, MD_NSAMPLES - 1);
                const int nd = t < MD_NSAMPLES ? t_nd[tt] : 0;
                // slot s = the trace's s-th domain from the left (the walk found them right to left)
                uint32_t ft[MD_MAXTDOM];
                float4 n2[MD_MAXTDOM];
#pragma unroll
                for (int sl = 0; sl < MD_MAXTDOM; sl++) {
                    const int d = nd - 1 - sl;
                    ft[sl] = 0u; n2[sl] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (d >= 0) { ft[sl] = t_ft[d * MD_NSAMPLES + tt]; n2[sl] = t_n2[d * MD_NSAMPLES + tt]; }
                }
                int inc = nd;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(FULL, inc, o);
                    if (lane >= o) inc += v;
                }
                const int at = inc - nd, count = __shfl_sync(FULL, inc, 31);
                __syncwarp();                      // the previous round has been read
#pragma unroll
                for (int sl = 0; sl < MD_MAXTDOM; sl++) {
                    if (sl < nd) {
                        st_ft[at + sl] = ft[sl];
                        st_n2[at + sl] = n2[sl];
                        if (first_pass) {
                            const uint32_t km = t_km[(nd - 1 - sl) * MD_NSAMPLES + tt];
                            const unsigned long long si = (ft[sl] & 0xffffu) + (uint32_t)(ireg - 1), sj = (ft[sl] >> 16) + (uint32_t)(ireg - 1);
                            rkey[nraw + at + sl] = (si & 0xffffu) | ((sj & 0xffffu) << 16) | ((unsigned long long)(km & 0xffffu) << 32);
                            rtr[nraw + at + sl] = (uint8_t)t;
                        }
                    }
                }
                if (first_pass) nraw += count;
                __syncwarp();
                if (plain) md_accumulate_nb<true>(nb, st_ft, st_n2, count, pg + lane, x, sum, cover);
                else md_accumulate_nb<false>(nb, st_ft, st_n2, count, pg + lane, x, sum, cover);
            }
#pragma unroll
            for (int b = 0; b < MDC_PB; b++) {
                const int pos = pg + 32 * b + lane;
                if (pos <= Ld) acc[pos] = logf_via_double((sum[b] + (float)(MD_NSAMPLES - cover[b])) / (float)MD_NSAMPLES);
            }
        }
        __syncwarp();
        for (int h = lane; h < MDC_HT; h += 32) sm.htab[h] = EMPTY;
        __syncwarp();
        // n2sc of the region: the sum in position order
        float regsum = 0.f;
        if (lane == 0)
            for (int pos = 1; pos <= Ld; pos++) regsum += acc[pos];
        // ---- B. distinct segments ----
        for (int q = lane; q < nraw; q += 32) {
            const unsigned long long key = rkey[q];
            uint32_t h = ((uint32_t)(key ^ (key >> 21)) * 0x9E3779B1u) >> 22;
            for (;;) {
                uint32_t cur = *(volatile uint32_t *)&sm.htab[h];
                if (cur == EMPTY) {
                    cur = atomicCAS(&sm.htab[h], EMPTY, (uint32_t)q);
                    if (cur == EMPTY) break;
                }
                if (rkey[cur] == key) { atomicMin(&sm.htab[h], (uint32_t)q); break; }
                h = (h + 1) & (MDC_HT - 1);
            }
            rslot[q] = (uint16_t)h;
        }
        __syncwarp();
        int nseg = 0;
        for (int q0 = 0; q0 < nraw; q0 += 32) {
            const int q = q0 + lane;
            uint32_t h = 0;
            bool first = false;
            if (q < nraw) { h = rslot[q]; first = sm.htab[h] == (uint32_t)q; }
            const unsigned m = __ballot_sync(FULL, first);
            if (first) {
                const int id = nseg + __popc(m & lt);
                sm.skey[id] = md_seg_word(rkey[q]);
                sm.scount[id] = 0u;
                sm.asg[id] = -1;
                sm.htab[h] = 0x80000000u | (uint32_t)id;
            }
            nseg += __popc(m);
        }
        __syncwarp();
        for (int q = lane; q < nraw; q += 32) {
            const uint32_t id = sm.htab[rslot[q]] & 0x7fffffffu;
            rslot[q] = (uint16_t)id;
            atomicAdd(&sm.scount[id], 1u);
        }
        __syncwarp();
        // ---- C. single linkage clustering over the DISTINCT segments (same components as over all samples) ----
        int nc = 0;
        for (int q = 0; q < nseg; q++) {
            if (sm.asg[q] >= 0) continue;
            __syncwarp();
            if (lane == 0) { sm.queue[0] = (int16_t)q; sm.asg[q] = (int16_t)nc; }
            __syncwarp();
            int head = 0, tail = 1;
            const int lo = q & ~31;                 // every segment below the seed already has its cluster
            while (head < tail) {
                int ntail = tail;
                for (int b0 = lo; b0 < nseg; b0 += 32) {
                    const int bb = b0 + lane;
                    bool take = false;
                    if (bb < nseg && sm.asg[bb] < 0) {
                        const unsigned long long kb = sm.skey[bb];
                        for (int f = head; f < tail && !take; f++) take = md_link_word(sm.skey[sm.queue[f]], kb);
                    }
                    const unsigned m = __ballot_sync(FULL, take);
                    if (take) {
                        sm.asg[bb] = (int16_t)nc;
                        sm.queue[ntail + __popc(m & lt)] = (int16_t)bb;
                    }
                    ntail += __popc(m);
                }
                __syncwarp();
                head = tail;
                tail = ntail;
            }
            nc++;
        }
        __syncwarp();
        // ---- D. traces per cluster (the samples of a trace are consecutive) ----
        for (int c = lane; c < nc; c += 32) sm.htab[c] = 0u;
        __syncwarp();
        for (int q = lane; q < nraw; q += 32) {
            const int c = sm.asg[rslot[q]], t = rtr[q];
            bool dup = false;
            for (int b = 1; b < MD_MAXTDOM && q - b >= 0 && !dup; b++) {
                if (rtr[q - b] != t) break;
                dup = sm.asg[rslot[q - b]] == c;
            }
            if (!dup) atomicAdd(&sm.htab[c], 1u);
        }
        __syncwarp();
        // clusters with posterior >= 0.25 (at most MD_NSAMPLES * MD_MAXTDOM / 50 = 16 of them), in cluster order
        int npass = 0;
        for (int c0 = 0; c0 < nc; c0 += 32) {
            const int c = c0 + lane;
            const bool ok = c < nc && !((float)sm.htab[c] / (float)MD_NSAMPLES < 0.25f);
            const unsigned m = __ballot_sync(FULL, ok);
            if (ok && npass + __popc(m & lt) < 16) sm.queue[npass + __popc(m & lt)] = (int16_t)c;
            npass = min(npass + __popc(m), 16);
        }
        __syncwarp();
        int ci[16], cj[16];
        int nenv = 0;
        for (int pc = 0; pc < npass; pc++) {
            const int c = sm.queue[pc];
            int ninc = 0;
            int imin = 1 << 30, imax = 0, jmin = 1 << 30, jmax = 0;
            for (int q = lane; q < nseg; q += 32) {
                if (sm.asg[q] != c) continue;
                const unsigned long long k = sm.skey[q];
                const int si = (int)(k & 0xffffu), sj = (int)((k >> 16) & 0xffffu);
                ninc += (int)sm.scount[q];
                imin = min(imin, si); imax = max(imax, si);
                jmin = min(jmin, sj); jmax = max(jmax, sj);
            }
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                ninc += __shfl_xor_sync(FULL, ninc, o);
                imin = min(imin, __shfl_xor_sync(FULL, imin, o)); imax = max(imax, __shfl_xor_sync(FULL, imax, o));
                jmin = min(jmin, __shfl_xor_sync(FULL, jmin, o)); jmax = max(jmax, __shfl_xor_sync(FULL, jmax, o));
            }
            const int thr = (int)ceilf((float)ninc * 0.02f);
            // leftmost start / rightmost end whose count reaches thr: histogram of the cluster's end points
            int best[2];
#pragma unroll
            for (int side = 0; side < 2; side++) {
                const int vmin = side ? jmin : imin, vmax = side ? jmax : imax, span = vmax - vmin + 1;
                int found = -1;
                for (int w0 = 0; w0 < span && found < 0; w0 += MDC_HT) {      // one window unless the span is huge
                    const int wn = min(span - w0, MDC_HT);
                    __syncwarp();
                    for (int h = lane; h < wn; h += 32) sm.htab[h] = 0u;
                    __syncwarp();
                    for (int q = lane; q < nseg; q += 32) {
                        if (sm.asg[q] != c) continue;
                        const unsigned long long k = sm.skey[q];
                        const int v = side ? (int)((k >> 16) & 0xffffu) : (int)(k & 0xffffu);
                        // the window counts from vmin upwards (starts) or from vmax downwards (ends)
                        const int off = (side ? vmax - v : v - vmin) - w0;
                        if (off >= 0 && off < wn) atomicAdd(&sm.htab[off], sm.scount[q]);
                    }
                    __syncwarp();
                    for (int h0 = 0; h0 < wn && found < 0; h0 += 32) {
                        const bool hit = h0 + lane < wn && (int)sm.htab[h0 + lane] >= thr;
                        const unsigned m = __ballot_sync(FULL, hit);
                        if (m) found = w0 + h0 + __ffs(m) - 1;
                    }
                }
                if (found < 0) found = span;                     // the reference loop runs off the end
                best[side] = side ? vmax - found : vmin + found;
            }
            const int best_i = best[0], best_j = best[1];
            if (nenv < 16) {
                int at = nenv;
                while (at > 0 && (ci[at - 1] > best_i || (ci[at - 1] == best_i && cj[at - 1] > best_j))) {
                    ci[at] = ci[at - 1]; cj[at] = cj[at - 1]; at--;
                }
                ci[at] = best_i; cj[at] = best_j;
                nenv++;
            }
        }
        if (lane == 0) {
            if (nenv > ITSX_MAXDOM) {
                atomicAdd(&a.counters[CNT_DOM_OVERFLOW], (unsigned long long)(nenv - ITSX_MAXDOM));
                nenv = ITSX_MAXDOM;
            }
            MdRes res;
            res.n = nenv; res.regsum = regsum;
            for (int c = 0; c < ITSX_MAXDOM; c++) { res.ci[c] = 0; res.cj[c] = 0; res.cdc[c] = 0.f; }
            for (int c = 0; c < nenv; c++) {
                float dc = 0.f;
                for (int pos = ci[c]; pos <= cj[c]; pos++) dc += acc[pos - ireg + 1];
                res.ci[c] = ci[c]; res.cj[c] = cj[c]; res.cdc[c] = dc;
            }
            a.res[r] = res;
        }
        __syncwarp();
    }
}

// number of flagged regions of every worklist entry
__global__ void mdcount_kernel(const uint8_t *__restrict__ ndom, const int32_t *__restrict__ env, int n,
                               int32_t *__restrict__ nreg)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e > n) return;
    int c = 0;
    if (e < n) {
        const int nd = ndom[e];
        for (int d = 0; d < nd; d++) c += (env[((size_t)e * ITSX_MAXDOM + d) * 2 + 1] >> 30) & 1;
    }
    nreg[e] = c;
}
// region list in entry order: entry, coordinates, rows of the slab (Ld + 1)
__global__ void mdregs_kernel(const uint8_t *__restrict__ ndom, const int32_t *__restrict__ env, int n,
                              const int32_t *__restrict__ base, int32_t *__restrict__ reg_ent,
                              int32_t *__restrict__ reg_i, int32_t *__restrict__ reg_j, int32_t *__restrict__ reg_rows)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    if (base[e + 1] == base[e]) return;
    const int nd = ndom[e];
    int at = base[e];
    for (int d = 0; d < nd; d++) {
        const int jraw = env[((size_t)e * ITSX_MAXDOM + d) * 2 + 1];
        if ((jraw >> 30) & 1) {
            const int i = env[((size_t)e * ITSX_MAXDOM + d) * 2 + 0], j = jraw & 0x1fffffff;
            reg_ent[at] = e; reg_i[at] = i; reg_j[at] = j; reg_rows[at] = j - i + 2;
            at++;
        }
    }
}
// the cluster envelopes replace the flagged regions in the entry's list
__global__ void mdapply_kernel(uint8_t *__restrict__ ndom, int32_t *__restrict__ env, int n,
                               const int32_t *__restrict__ base, const MdRes *__restrict__ res,
                               float *__restrict__ envdc, float *__restrict__ n2reg,
                               unsigned long long *__restrict__ counters)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    if (base[e + 1] == base[e]) return;
    const int nd = ndom[e];
    int oi[ITSX_MAXDOM], oj[ITSX_MAXDOM];
    for (int d = 0; d < nd; d++) {
        oi[d] = env[((size_t)e * ITSX_MAXDOM + d) * 2 + 0];
        oj[d] = env[((size_t)e * ITSX_MAXDOM + d) * 2 + 1];
    }
    int nn = 0, at = base[e];
    float n2sum = 0.f;
    for (int d = 0; d < nd; d++) {
        if (!((oj[d] >> 30) & 1)) {
            if (nn < ITSX_MAXDOM) {
                env[((size_t)e * ITSX_MAXDOM + nn) * 2 + 0] = oi[d];
                env[((size_t)e * ITSX_MAXDOM + nn) * 2 + 1] = oj[d];
                envdc[(size_t)e * ITSX_MAXDOM + nn] = 0.f;
                nn++;
            }
            continue;
        }
        const MdRes rs = res[at++];
        n2sum += rs.regsum;
        for (int c = 0; c < rs.n; c++) {
            if (nn < ITSX_MAXDOM) {
                env[((size_t)e * ITSX_MAXDOM + nn) * 2 + 0] = rs.ci[c];
                env[((size_t)e * ITSX_MAXDOM + nn) * 2 + 1] = rs.cj[c] | (1 << 30) | (1 << 29);
                envdc[(size_t)e * ITSX_MAXDOM + nn] = rs.cdc[c];
                nn++;
            } else {
                atomicAdd(&counters[CNT_DOM_OVERFLOW], 1ull);
            }
        }
    }
    ndom[e] = (uint8_t)nn;
    n2reg[e] = n2sum;
}

// ------------------------------------------------------------------------------------------------
// envelope worklist
__global__ void ndom_widen_kernel(const uint8_t *__restrict__ ndom, int n, int32_t *__restrict__ out)
{
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n) out[e] = ndom[e];
    if (e == n) out[e] = 0;
}
// work item = entry * MAXDOM + d; sort key = (profile, envelope length) so that the 32 envelopes of a warp tile
// have (nearly) the same number of rows -- lanes of a tile run to the longest envelope
__global__ void envwork_kernel(const uint8_t *__restrict__ ndom, const int32_t *__restrict__ envoff, int n,
                               const int32_t *__restrict__ list, int ns, const int32_t *__restrict__ env,
                               int32_t *__restrict__ work, uint32_t *__restrict__ key)
{
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int nd = ndom[e], o = envoff[e];
    const uint32_t p = (uint32_t)(list[e] / ns);
    for (int d = 0; d < nd; d++) {
        const int ienv = env[((size_t)e * ITSX_MAXDOM + d) * 2 + 0];
        const int jenv = env[((size_t)e * ITSX_MAXDOM + d) * 2 + 1] & 0x1fffffff;
        work[o + d] = e * ITSX_MAXDOM + d;
        key[o + d] = (p << 12) | (uint32_t)min(jenv - ienv + 1, 4095);
    }
}
__global__ void gather_bounds_kernel(const int32_t *__restrict__ envoff, const int32_t *__restrict__ bounds, int P,
                                     int32_t *__restrict__ out)
{
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p <= P) out[p] = envoff[bounds[p]];
}

// K10: envelope rescoring (unihit Forward, Backward, posterior decoding, null2 by expectation)
struct EnvArgs {
    const int32_t *work;      // this profile's slice of the envelope worklist: entry*MAXDOM + d
    int            count;
    const int32_t *list;      // whole pair list of the batch
    const int32_t *envoff;    // first envelope number of every entry (output slot = envoff[entry] + d)
    const int32_t *env;
    const int32_t *order;
    int64_t        s0;
    int            ns, prof;
    const uint32_t *seqw;
    const int64_t  *woff;
    const int32_t  *seqlen;
    const float    *etab;
    float          *scratch;  // warps_total * (Ldmax+1) * ENV_ROWF * 32 floats (match rows + raw E)
    int             Ldmax;
    float          *out;      // [envelope][20]: envsc, domcorrection, null2[16], pad
    int             out_base; // index of this slice's first envelope in the batch numbering
    unsigned long long *counters;
};

__global__ void __launch_bounds__(ENV_THREADS, ENV_CTAS_PER_SM)
env_kernel(const __grid_constant__ ProfConst pc, const EnvArgs a)
{
    __shared__ __align__(16) float s_e[16 * ESTRIDE];     // [residue code][node]: odds of the launch's profile
    for (int t = threadIdx.x; t < 16 * ESTRIDE; t += ENV_THREADS) {
        const int x = t / ESTRIDE, k = t - x * ESTRIDE;
        s_e[t] = k <= MAXM ? a.etab[k * 16 + x] : 0.f;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int wid = threadIdx.x >> 5;
    const int warp_in_grid = (blockIdx.x * ENV_THREADS + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * ENV_THREADS) >> 5;
    const int ntiles = (a.count + 31) >> 5;
    float *sc = a.scratch + (size_t)warp_in_grid * (size_t)(a.Ldmax + 1) * ENV_ROWF * 32 + lane;
#define ROW(row, c) sc[((size_t)(row) * ENV_ROWF + (c)) * 32]
    // Backward reads the Forward rows back in reverse order: each warp streams its rows (ENV_ROWBYTES, contiguous)
    // into a two-deep shared-memory ring with bulk async copies, one row ahead of use.
    extern __shared__ __align__(128) unsigned char env_smem[];
    float *ring = (float *)env_smem + (size_t)wid * ENV_RING * ENV_ROWF * 32;
    unsigned long long *bars = (unsigned long long *)(env_smem + (size_t)(ENV_THREADS / 32) * ENV_RING * ENV_ROWBYTES) + wid * ENV_RING;
    const uint32_t bar0 = smem_u32(bars), ring0 = smem_u32(ring);
    if (lane == 0) {
#pragma unroll
        for (int b = 0; b < ENV_RING; b++) mbar_init(bar0 + b * 8, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncwarp();
    uint32_t phases = 0u;                      // bit b: parity the next wait on slot b expects
    const float *rowbase = a.scratch + (size_t)warp_in_grid * (size_t)(a.Ldmax + 1) * ENV_ROWF * 32;
    constexpr int C_E = MAXM;

    for (int tile = warp_in_grid; tile < ntiles; tile += nwarps) {
        const int t = tile * 32 + lane;
        const bool valid = t < a.count;
        int L = 0, Ld = 0, ienv = 1, oslot = 0;
        const uint32_t *w = a.seqw;
        if (valid) {
            const int wk = a.work[t];
            const int ent = wk / ITSX_MAXDOM, d = wk - ent * ITSX_MAXDOM;
            oslot = a.envoff[ent] + d;
            const int idx = a.list[ent];
            const int sl = idx - a.prof * a.ns;
            const int64_t s = a.order[a.s0 + sl];
            L = a.seqlen[s];
            w = a.seqw + a.woff[s];
            ienv = a.env[((size_t)ent * ITSX_MAXDOM + d) * 2 + 0];
            const int jenv = a.env[((size_t)ent * ITSX_MAXDOM + d) * 2 + 1] & 0x1fffffff;
            Ld = jenv - ienv + 1;
        }
        int Lw = Ld;
#pragma unroll
        for (int o = 16; o; o >>= 1) Lw = max(Lw, __shfl_xor_sync(0xffffffffu, Lw, o));

        // unihit length model for the full target length (nj = 0)
        const float pmove = (2.0f + 0.0f) / ((float)L + 2.0f + 0.0f);
        const float N_move = pmove, N_loop = 1.0f - pmove;
        const float E_move = 1.0f, E_loop = 0.0f;

        float Mx[MAXM + 2], Ix[MAXM + 2], Dx[MAXM + 2];
#pragma unroll
        for (int k = 0; k <= MAXM + 1; k++) Mx[k] = Ix[k] = Dx[k] = 0.f;

        // ---- Forward over the envelope; match rows (+ raw E) go to the scratch slab ----
        float xN = 1.f, xJ = 0.f, xC = 0.f, xE = 0.f, xB = N_move, totscale = 0.f;
        for (int i = 1; i <= Lw; i++) {
            if (i <= Ld) {
                const float4 *er = (const float4 *)(s_e + residue_at(w, ienv - 1 + i - 1) * ESTRIDE);
                // pass 1, descending k, in place: M and I of row i from row i-1 (no serial dependence, so the
                // scheduler needs no far-ahead coefficient loads); pass 2, ascending: the D chain and the E sums.
                // Same operations and summation order as the oracle's single ascending loop.
#pragma unroll
                for (int k = MAXM; k >= 1; k--) {
                    float sv = xB * pc.fa[k][0];
                    sv = fmaf(Mx[k - 1], pc.fa[k][1], sv);
                    sv = fmaf(Ix[k - 1], pc.fa[k][2], sv);
                    sv = fmaf(Dx[k - 1], pc.fa[k][3], sv);
                    sv = sv * EMIS(er, k);
                    const float ic = fmaf(Ix[k], pc.fi[k][0], Mx[k] * pc.fi[k][1]);
                    Mx[k] = sv; Ix[k] = ic;
                }
                float xEm = 0.f, xEd = 0.f, dcur = 0.f;
#pragma unroll
                for (int k = 1; k <= MAXM; k++) {
                    const float dc = fmaf(dcur, pc.fd[k][0], Mx[k - 1] * pc.fd[k][1]);
                    Dx[k] = dc; dcur = dc;
                    xEm += Mx[k]; xEd += dc;
                }
                xE = xEm + xEd;
                xN = xN * N_loop;
                xC = fmaf(xC, N_loop, xE * E_move);
                xJ = fmaf(xJ, N_loop, xE * E_loop);
                xB = fmaf(xJ, N_move, xN * N_move);
                const float eraw = xE;
                if (xE > 1.0e4f) {
                    xN = xN / xE; xC = xC / xE; xJ = xJ / xE; xB = xB / xE;
                    const float inv = 1.0f / xE;
#pragma unroll
                    for (int k = 1; k <= MAXM; k++) { Mx[k] *= inv; Dx[k] *= inv; Ix[k] *= inv; }
                    totscale += logf_via_double(xE);
                    xE = 1.0f;
                }
#pragma unroll
                for (int k = 1; k <= MAXM; k++) ROW(i, k - 1) = Mx[k];
                ROW(i, C_E) = eraw;
            }
        }
        const float envsc = totscale + logf_via_double(xC * N_move);

        // ---- Backward; nk[k] accumulates the expected usage of match state k ----
        float nk[MAXM + 1];
#pragma unroll
        for (int k = 0; k <= MAXM; k++) nk[k] = 0.f;
        float bJ = 0.f, bB = 0.f, bN = 0.f, bC = N_move, bE = bC * E_move;
        if (valid) {
            Dx[MAXM + 1] = 0.f;
#pragma unroll
            for (int k = MAXM; k >= 1; k--) {
                Dx[k] = fmaf(pc.bd1[k - 1], Dx[k + 1], bE);
                Mx[k] = fmaf(pc.bd2[k - 1], Dx[k + 1], bE);
                Ix[k] = 0.f;
            }
            float fE, fS;
            spec_decode(ROW(Ld, C_E), fE, fS);
            if (fS > 1.0f) {
                bE = bE / fS; bN = bN / fS; bC = bC / fS; bJ = bJ / fS; bB = bB / fS;
                const float inv = 1.0f / fS;
#pragma unroll
                for (int k = 1; k <= MAXM; k++) { Mx[k] *= inv; Dx[k] *= inv; Ix[k] *= inv; }
            }
        }
        // the rows were written through the generic proxy; order them before the async-proxy reads
        asm volatile("fence.proxy.async;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
#pragma unroll
            for (int d = 0; d < ENV_RING; d++) {
                const int row = Lw - d;
                if (row >= 1)
                    tma_row_load(ring0 + (row & (ENV_RING - 1)) * ENV_ROWBYTES, rowbase + (size_t)row * ENV_ROWF * 32, ENV_ROWBYTES,
                                 bar0 + (row & (ENV_RING - 1)) * 8);
            }
        }
        // raw E of row i-1 (rescale of the new Backward row) comes through a register, one row ahead
        float qE = (Lw >= 2 && Lw - 1 <= Ld) ? ROW(Lw - 1, C_E) : 0.f;
        for (int i = Lw; i >= 1; i--) {
            const int b = i & (ENV_RING - 1);
            mbar_wait(bar0 + b * 8, (phases >> b) & 1u);
            phases ^= 1u << b;
            const float *rs = ring + (size_t)b * ENV_ROWF * 32 + lane;
            const float cEp = qE;
            if (i >= 3 && i - 2 <= Ld) qE = ROW(i - 2, C_E);
            if (i <= Ld) {
                float fE, fS;
                spec_decode(rs[C_E * 32], fE, fS);
#pragma unroll
                for (int k = 1; k <= MAXM; k++) nk[k] = fmaf(rs[(k - 1) * 32] * Mx[k], fS, nk[k]);
            }
            __syncwarp();
            if (lane == 0 && i > ENV_RING)
                tma_row_load(ring0 + b * ENV_ROWBYTES, rowbase + (size_t)(i - ENV_RING) * ENV_ROWF * 32, ENV_ROWBYTES, bar0 + b * 8);
            if (i <= Ld) {
                if (i > 1) {
                    float fEp, fSp;
                    spec_decode(cEp, fEp, fSp);
                    const float4 *er = (const float4 *)(s_e + residue_at(w, ienv - 1 + i - 1) * ESTRIDE);
                    bB = 0.f;
#pragma unroll
                    for (int k = 1; k <= MAXM; k++) {
                        Mx[k] = Mx[k] * EMIS(er, k);
                        bB = fmaf(Mx[k], pc.bm[k - 1], bB);
                    }
                    bC = bC * N_loop;
                    bJ = fmaf(bB, N_move, bJ * N_loop);
                    bN = fmaf(bB, N_move, bN * N_loop);
                    bE = fmaf(bC, E_move, bJ * E_loop);
                    Dx[MAXM + 1] = 0.f;
                    float mnext = 0.f;
#pragma unroll
                    for (int k = MAXM; k >= 1; k--) {
                        const float mpe_k = Mx[k];
                        const float ic = fmaf(mnext, pc.ba[k][0], Ix[k] * pc.ba[k][1]);
                        // every M and D state also exits to E: bE is the addend the FMA chains start from
                        const float dc = fmaf(mnext, pc.bd0[k - 1], fmaf(Dx[k + 1], pc.bd1[k - 1], bE));
                        const float mc = fmaf(mnext, pc.ba[k][2], fmaf(Ix[k], pc.ba[k][3], fmaf(Dx[k + 1], pc.bd2[k - 1], bE)));
                        Mx[k] = mc; Ix[k] = ic; Dx[k] = dc;
                        mnext = mpe_k;
                    }
                    if (fSp > 1.0f) {
                        bE = bE / fSp; bN = bN / fSp; bC = bC / fSp; bJ = bJ / fSp; bB = bB / fSp;
                        const float inv = 1.0f / fSp;
#pragma unroll
                        for (int k = 1; k <= MAXM; k++) { Mx[k] *= inv; Dx[k] *= inv; Ix[k] *= inv; }
                    }
                } else {
                    const float4 *er = (const float4 *)(s_e + residue_at(w, ienv - 1) * ESTRIDE);
                    bB = 0.f;
#pragma unroll
                    for (int k = 1; k <= MAXM; k++) bB = fmaf(Mx[k] * EMIS(er, k), pc.bm[k - 1], bB);
                    bN = fmaf(bB, N_move, bN * N_loop);
                }
            }
        }
        if (valid) {
            // null2[x] = 1 + sum_k pbar(M_k) (odds_k[x] - 1): every non-match emitter has odds 1 (see oracle)
            const float scaleproduct = 1.0f / bN;
            const float norm = 1.0f / (float)Ld;
            float null2[16];
#pragma unroll
            for (int x = 0; x < 4; x++) {
                float ws = 0.f;
#pragma unroll
                for (int k = 1; k <= MAXM; k++) ws = fmaf(nk[k], s_e[x * ESTRIDE + k] - 1.0f, ws);
                null2[x] = 1.0f + ws * scaleproduct * norm;
            }
            const int degen[16] = {1, 2, 4, 8, 5, 10, 3, 12, 6, 9, 11, 14, 7, 13, 15, 0};
#pragma unroll
            for (int x = 4; x < 15; x++) {
                float s = 0.f;
                int n = 0;
#pragma unroll
                for (int y = 0; y < 4; y++)
                    if (degen[x] & (1 << y)) { s += null2[y]; n++; }
                null2[x] = s / (float)n;
            }
            null2[15] = 1.0f;
            float *o = a.out + (size_t)oslot * 20;
            o[0] = envsc;
#pragma unroll
            for (int x = 0; x < 16; x++) o[2 + x] = null2[x];
            atomicAdd(&a.counters[CNT_ENV_ROWS], (unsigned long long)Ld);
            atomicMax(&a.counters[CNT_MAX_ENVLEN], (unsigned long long)Ld);
        }
    }
#undef ROW
}

// ------------------------------------------------------------------------------------------------
// the "%6.1f"-printed score in integer tenths, and ItsPosition's ordering key under max: (score10, NOT row rank) --
// row order of the reference table restricted to one target = (profile, domain index), first row wins ties
__device__ __forceinline__ int score10_of(float bits) { return (int)rint((double)bits * 10.0); }
__device__ __forceinline__ unsigned long long row_key(float bits, int prof, int dom_idx)
{
    const unsigned long long sc = (unsigned long long)(score10_of(bits) + (1 << 20));
    const unsigned long long rank = (unsigned long long)prof * ITSX_MAXDOM + (unsigned long long)dom_idx;
    return (sc << 40) | (0xFFFFFFFFFFull - rank);
}

// K11a: per-hit and per-domain scores (SURVEY A.4 steps 6-7), -T threshold, reported-hit counts
struct FinalArgs {
    const int32_t *list;
    int            n;         // entries in the batch
    const int32_t *order;
    int64_t        s0;
    int            ns;
    const uint32_t *seqw;
    const int64_t  *woff;
    const int32_t  *seqlen;
    const ProfScalars *pscal;
    const float    *nullsctab;
    const float    *logsum;
    const float    *fwdsc;
    const uint8_t  *ndom;
    const int32_t  *envoff;
    const int32_t  *env;
    const float    *envdc;    // [entry][MAXDOM]: domcorrection of the envelopes whose null2 came from traces (bit 29)
    const float    *n2reg;    // [entry]: trace n2sc summed over the entry's multidomain regions
    float          *envout;   // [envelope][20]; [1] receives domcorrection
    float           T;
    DomRec         *doms;     // output base for this batch (keep_rows mode 1)
    int32_t        *nrep;     // per (sample, profile)
    const int32_t  *seq_sample;   // sample of every searched sequence (NULL: one sample)
    int             P;
    unsigned long long *counters;
    // compact mode (keep_rows 2): rows that are printed whatever domZ turns out to be enter the arg-max at once
    int             compact;
    unsigned long long *best; // [2][nseq]
    int64_t         nseq, seq_first;
    double          lnP_certain;   // ln(domE / domz_upper): lnP <= this  =>  P x domZ <= domE for every possible domZ
};

__global__ void __launch_bounds__(128) final_kernel(const FinalArgs a)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.n) return;
    const int nd = a.ndom[e];
    if (nd == 0) return;
    const int idx = a.list[e];
    const int p = idx / a.ns, sl = idx - p * a.ns;
    const int64_t s = a.order[a.s0 + sl];
    const int L = a.seqlen[s];
    const uint32_t *w = a.seqw + a.woff[s];
    const ProfScalars &ps = a.pscal[p];
    const float nullsc = a.nullsctab[L];
    const float fwdsc = a.fwdsc[e];
    const int o0 = a.envoff[e];
    const float omega = 1.0f / 256.0f;
    const float lnomega = logf_via_double(omega);

    // n2sc summed over the whole sequence (position order) and per envelope
    float seqbias = 0.f;
    for (int d = 0; d < nd; d++) {
        float *o = a.envout + (size_t)(o0 + d) * 20;
        const int ienv = a.env[((size_t)e * ITSX_MAXDOM + d) * 2 + 0];
        const int jraw = a.env[((size_t)e * ITSX_MAXDOM + d) * 2 + 1];
        const int jenv = jraw & 0x1fffffff;
        if ((jraw >> 29) & 1) {         // null2 by trace: the whole region counts once, below
            o[1] = a.envdc[(size_t)e * ITSX_MAXDOM + d];
            continue;
        }
        float dc = 0.f;
        for (int pos = ienv; pos <= jenv; pos++) {
            const float v = logf(o[2 + residue_at(w, pos - 1)]);
            dc += v;
            seqbias += v;
        }
        o[1] = dc;
    }
    seqbias += a.n2reg[e];
    seqbias = flogsum(a.logsum, 0.0f, lnomega + seqbias);
    float pre_score = (float)((double)(fwdsc - nullsc) / kLn2);
    float sscore = (float)((double)(fwdsc - (nullsc + seqbias)) / kLn2);
    float sum_score = 0.0f, sbias = 0.0f;
    int Ldsum = 0;
    for (int d = 0; d < nd; d++) {
        const float *o = a.envout + (size_t)(o0 + d) * 20;
        if (o[0] - o[1] > 0.0f) {
            const int ienv = a.env[((size_t)e * ITSX_MAXDOM + d) * 2 + 0];
            const int jenv = a.env[((size_t)e * ITSX_MAXDOM + d) * 2 + 1] & 0x1fffffff;
            sum_score += o[0];
            Ldsum += jenv - ienv + 1;
            sbias += o[1];
        }
    }
    sbias = flogsum(a.logsum, 0.0f, lnomega + sbias);
    const double lratio = log((double)((float)L / (float)(L + 3)));
    sum_score += (float)((L - Ldsum) * lratio);
    float pre2 = (float)((double)(sum_score - nullsc) / kLn2);
    sum_score = (float)((double)(sum_score - (nullsc + sbias)) / kLn2);
    if (Ldsum > 0 && sum_score > sscore) { sscore = sum_score; pre_score = pre2; }
    (void)pre_score;
    const double seq_lnP = exp_logsurv((double)sscore, (double)ps.ev[EV_FTAU], (double)ps.ev[EV_FLAMBDA]);
    const int reported = sscore >= a.T;
    if (reported) {
        atomicAdd(&a.nrep[(a.seq_sample ? (size_t)a.seq_sample[s] * a.P : 0) + p], 1);
        atomicAdd(&a.counters[CNT_HITS_REPORTED], 1ull);
    }
    for (int d = 0; d < nd; d++) {
        float *o = a.envout + (size_t)(o0 + d) * 20;
        const int ienv = a.env[((size_t)e * ITSX_MAXDOM + d) * 2 + 0];
        const int jraw = a.env[((size_t)e * ITSX_MAXDOM + d) * 2 + 1];
        const int jenv = jraw & 0x1fffffff;
        const int ld = jenv - ienv + 1;
        const float bs = o[0] + (float)((L - ld) * lratio);
        const float dombias = flogsum(a.logsum, 0.0f, lnomega + o[1]);
        const float bitscore = (float)((double)(bs - (nullsc + dombias)) / kLn2);
        const double lnP = exp_logsurv((double)bitscore, (double)ps.ev[EV_FTAU], (double)ps.ev[EV_FLAMBDA]);
        if (a.compact) {
            // bit 0: the hit is reported (-T); bit 1: the row is printed for every possible domZ
            const int certain = reported && lnP <= a.lnP_certain;
            o[18] = bitscore;
            o[19] = __int_as_float(reported | (certain << 1));
            o[17] = sscore;
            if (certain) {
                atomicAdd(&a.counters[CNT_CERTAIN], 1ull);
                if (ps.side >= 0)
                    atomicMax(&a.best[(size_t)ps.side * a.nseq + (s - a.seq_first)], row_key(bitscore, p, d));
            }
            continue;
        }
        DomRec r;
        r.seq = (int32_t)s; r.prof = p; r.ienv = ienv; r.jenv = jenv; r.tlen = L; r.dom_idx = d;
        r.bitscore = bitscore;
        r.envsc = o[0]; r.domcorrection = o[1]; r.seq_score = sscore;
        r.lnP = lnP;
        r.seq_lnP = seq_lnP;
        r.is_multidomain = (jraw >> 30) & 1;
        r.pair_reported = reported;
        a.doms[o0 + d] = r;
    }
}

// compact mode, second pass over the batch once every certain row has entered the arg-max: the certain winners leave
// their coordinates in the position table; an undecided row is kept (appended to doms) only if it would beat the
// certain winner of its (sequence, side) -- nothing else can change the outcome once domZ is known.
__global__ void __launch_bounds__(128) compact_select_kernel(const FinalArgs a, unsigned long long *__restrict__ ndom_at,
                                                            int32_t *__restrict__ pos, uint8_t *__restrict__ selmulti)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.n) return;
    const int nd = a.ndom[e];
    if (nd == 0) return;
    const int idx = a.list[e];
    const int p = idx / a.ns, sl = idx - p * a.ns;
    const int64_t s = a.order[a.s0 + sl];
    const ProfScalars &ps = a.pscal[p];
    const int side = ps.side;
    const int o0 = a.envoff[e];
    const int64_t q = s - a.seq_first;
    for (int d = 0; d < nd; d++) {
        const float *o = a.envout + (size_t)(o0 + d) * 20;
        const int fl = __float_as_int(o[19]);
        if (!(fl & 1)) continue;                       // hit below -T: never printed
        const float bitscore = o[18];
        const int ienv = a.env[((size_t)e * ITSX_MAXDOM + d) * 2 + 0];
        const int jraw = a.env[((size_t)e * ITSX_MAXDOM + d) * 2 + 1];
        const int jenv = jraw & 0x1fffffff;
        const int multi = (jraw >> 30) & 1;
        if (side < 0) continue;                        // printed or not, ItsPosition ignores the row
        const unsigned long long key = row_key(bitscore, p, d);
        const unsigned long long cur = a.best[(size_t)side * a.nseq + q];
        if (fl & 2) {
            if (cur != key) continue;
            int32_t *b = pos + (size_t)(3 + 3 * side) * a.nseq;
            b[q] = score10_of(bitscore);
            b[a.nseq + q] = ienv;
            b[2 * a.nseq + q] = jenv;
            pos[2 * a.nseq + q] = a.seqlen[s];
            if (side == 0) pos[q] = jenv;
            else pos[a.nseq + q] = ienv - 1;
            selmulti[(size_t)side * a.nseq + q] = (uint8_t)multi;
        } else if (key > cur) {
            DomRec r;
            r.seq = (int32_t)s; r.prof = p; r.ienv = ienv; r.jenv = jenv; r.tlen = a.seqlen[s]; r.dom_idx = d;
            r.bitscore = bitscore; r.envsc = o[0]; r.domcorrection = o[1]; r.seq_score = o[17];
            r.lnP = exp_logsurv((double)bitscore, (double)ps.ev[EV_FTAU], (double)ps.ev[EV_FLAMBDA]);
            r.seq_lnP = exp_logsurv((double)o[17], (double)ps.ev[EV_FTAU], (double)ps.ev[EV_FLAMBDA]);
            r.is_multidomain = multi;
            r.pair_reported = 1;
            a.doms[atomicAdd(ndom_at, 1ull)] = r;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K11b + K12: domE threshold with the global domZ, then ItsPosition's arg-max.
// Row order of the reference table restricted to one target = (profile, domain index); the first row
// wins ties on the printed score, so the key is (score10, NOT rank) under max.
__global__ void select_kernel(DomRec *__restrict__ doms, int64_t n, const int32_t *__restrict__ nrep,
                              const int32_t *__restrict__ seq_sample, int P,
                              const ProfScalars *__restrict__ pscal, double domE,
                              unsigned long long *__restrict__ best, int64_t nseq, int64_t seq_first,
                              unsigned long long *__restrict__ counters)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    DomRec &r = doms[t];
    const int domZ = nrep[(seq_sample ? (size_t)seq_sample[r.seq] * P : 0) + r.prof];
    const int rep = r.pair_reported && (exp(r.lnP) * (double)domZ <= domE);
    r.pair_reported = rep ? 3 : (r.pair_reported & 1);   // bit1: row is printed
    if (!rep) return;
    atomicAdd(&counters[CNT_DOM_REPORTED], 1ull);
    const int side = pscal[r.prof].side;
    if (side < 0) return;
    atomicMax(&best[(size_t)side * nseq + (r.seq - seq_first)], row_key(r.bitscore, r.prof, r.dom_idx));
}

__global__ void best_kernel(const DomRec *__restrict__ doms, int64_t n, const ProfScalars *__restrict__ pscal,
                            const unsigned long long *__restrict__ best, int64_t nseq, int64_t seq_first,
                            int32_t *__restrict__ pos, uint8_t *__restrict__ selmulti)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const DomRec &r = doms[t];
    if (!(r.pair_reported & 2)) return;
    const int side = pscal[r.prof].side;
    if (side < 0) return;
    const unsigned long long key = row_key(r.bitscore, r.prof, r.dom_idx);
    const int64_t q = r.seq - seq_first;
    if (best[(size_t)side * nseq + q] != key) return;
    selmulti[(size_t)side * nseq + q] = (uint8_t)(r.is_multidomain != 0);
    int32_t *b = pos + (size_t)(3 + 3 * side) * nseq;
    b[q] = score10_of(r.bitscore);
    b[nseq + q] = r.ienv;
    b[2 * nseq + q] = r.jenv;
    pos[2 * nseq + q] = r.tlen;
    if (side == 0) pos[q] = r.jenv;             // start = left.to_pos            (SeqSample.py:480)
    else pos[nseq + q] = r.ienv - 1;            // stop  = right.from_pos - 1      (SeqSample.py:484)
}

__global__ void selmulti_count_kernel(const uint8_t *__restrict__ selmulti, int64_t n, unsigned long long *__restrict__ counters)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int v = t < n ? selmulti[t] : 0;
    const unsigned m = __ballot_sync(0xffffffffu, v != 0);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&counters[CNT_SEL_MULTI], (unsigned long long)__popc(m));
}

__global__ void pos_init_kernel(int32_t *pos, unsigned long long *best, uint8_t *selmulti, int64_t nseq)
{
    int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nseq) return;
    selmulti[q] = selmulti[nseq + q] = 0;
    pos[q] = pos[nseq + q] = pos[2 * nseq + q] = -1;
    pos[3 * nseq + q] = pos[6 * nseq + q] = INT32_MIN;
    pos[4 * nseq + q] = pos[5 * nseq + q] = pos[7 * nseq + q] = pos[8 * nseq + q] = -1;
    best[q] = best[nseq + q] = 0ull;
}

// esl_randomness_Init for the "fast" generator: the state after seeding (Jenkins mix3 of the seed)
uint32_t md_rng_state0(uint32_t seed)
{
    uint32_t a = seed, b = 87654321u, c = 12345678u;
    a -= b; a -= c; a ^= (c >> 13);
    b -= c; b -= a; b ^= (a << 8);
    c -= a; c -= b; c ^= (b >> 13);
    a -= b; a -= c; a ^= (c >> 12);
    b -= c; b -= a; b ^= (a << 16);
    c -= a; c -= b; c ^= (b >> 5);
    a -= b; a -= c; a ^= (c >> 3);
    b -= c; b -= a; b ^= (a << 10);
    c -= a; c -= b; c ^= (b >> 15);
    return c ? c : 42u;
}

// state after k more draws of x <- 69069 x + 1: x_(n+k) = A x_n + C (mod 2^32), by doubling
uint32_t md_rng_jump(uint32_t x, uint64_t k)
{
    uint32_t A = 1u, C = 0u, a = 69069u, cc = 1u;
    while (k) {
        if (k & 1u) { A = A * a; C = C * a + cc; }
        cc = cc * (a + 1u);
        a = a * a;
        k >>= 1;
    }
    return A * x + C;
}

}  // namespace

// ==================================================================================================
// host orchestration
// ==================================================================================================
int search_upload_profiles(itsx_ctx *c)
{
    if (!c->prof_dirty) return ITSX_OK;
    const int P = (int)c->prof.size();
    cudaStream_t st = c->stream;
    std::vector<uint32_t> msvtab((size_t)std::max(P, 1) * MSV_TABW);
    std::vector<float> etab((size_t)std::max(P, 1) * (MAXM + 1) * 16, 0.f);
    std::vector<ProfScalars> ps((size_t)std::max(P, 1));
    std::vector<float> mdtab((size_t)std::max(P, 1) * (MAXM + 2) * 8, 0.f);
    c->pconst.assign((size_t)P, ProfConst{});
    for (int p = 0; p < P; p++) {
        const HostProfile &h = c->prof[p];
        if (h.M > MAXM) {
            c->err = "profile '" + h.name + "' has more than ITSX_MAXM match states";
            return ITSX_ELIMIT;
        }
        if (h.bias_b >= 60) {
            c->err = "profile '" + h.name + "': MSV bias outside the range the s16x2 kernel is exact for";
            return ITSX_ELIMIT;
        }
        // layout A: word j = nodes (2j+1, 2j+2); layout B: word j = nodes (2j, 2j+1); absent nodes get -20000
        for (int lay = 0; lay < 2; lay++)
            for (int j = 0; j < KP; j++)
                for (int x = 0; x < 16; x++) {
                    int v[2];
                    for (int q = 0; q < 2; q++) {
                        const int k = 2 * j + q + (lay == 0 ? 1 : 0);
                        v[q] = (k >= 1 && k <= h.M) ? h.bias_b - (int)h.cost[k * 16 + x] : -20000;
                    }
                    msvtab[(size_t)p * MSV_TABW + ((size_t)lay * KP + j) * 16 + x] =
                        ((uint32_t)(uint16_t)(int16_t)v[0]) | ((uint32_t)(uint16_t)(int16_t)v[1] << 16);
                }
        for (int k = 1; k <= h.M; k++)
            for (int x = 0; x < 16; x++) etab[((size_t)p * (MAXM + 1) + k) * 16 + x] = h.e[k * 16 + x];
        ProfConst &pc = c->pconst[p];
        memset(&pc, 0, sizeof(pc));
        float tp[MAXM + 2][8];      // transitions out of node k (zero beyond the model), B->M_k entry in slot T_BM
        memset(tp, 0, sizeof(tp));
        for (int k = 0; k <= h.M; k++) {
            for (int s = 0; s < 7; s++) tp[k][s] = h.tp[k * 7 + s];
            tp[k][T_BM] = h.bm[k];
        }
        for (int k = 1; k <= MAXM; k++) {
            pc.fa[k][0] = tp[k][T_BM];
            pc.fa[k][1] = tp[k - 1][T_MM]; pc.fa[k][2] = tp[k - 1][T_IM]; pc.fa[k][3] = tp[k - 1][T_DM];
            pc.fi[k][0] = tp[k][T_II];     pc.fi[k][1] = tp[k][T_MI];
            pc.fd[k][0] = tp[k - 1][T_DD]; pc.fd[k][1] = tp[k - 1][T_MD];
            pc.ba[k][0] = tp[k][T_IM]; pc.ba[k][1] = tp[k][T_II]; pc.ba[k][2] = tp[k][T_MM]; pc.ba[k][3] = tp[k][T_MI];
            pc.bd0[k - 1] = tp[k][T_DM]; pc.bd1[k - 1] = tp[k][T_DD]; pc.bd2[k - 1] = tp[k][T_MD];
            pc.bm[k - 1] = tp[k][T_BM];
        }
        for (int k = 0; k <= MAXM + 1; k++)
            for (int t8 = 0; t8 < 8; t8++) mdtab[((size_t)p * (MAXM + 2) + k) * 8 + t8] = tp[k][t8];
        ProfScalars &q = ps[p];
        memset(&q, 0, sizeof(q));
        q.M = h.M; q.bias = h.bias_b; q.base = h.base_b; q.tbm = h.tbm_b; q.tec = h.tec_b;
        q.side = (p < (int)c->side.size()) ? c->side[p] : -1;
        q.scale_b = h.scale_b;
        for (int i = 0; i < 6; i++) q.ev[i] = h.ev[i];
        for (int x = 0; x < 16; x++) { q.eo[x][0] = h.eo[x][0]; q.eo[x][1] = h.eo[x][1]; }
    }
    // Viterbi filter tables (oracle/ora_hmm.c:viterbi_filter; HMMER p7_oprofile word scores): wordify(ln p), -32768 = -inf
    {
        auto wordify = [](float sc) -> int32_t {
            const float scale_w = 500.0f / (float)kLn2;
            if (!(sc > -INFINITY)) return -32768;
            sc = roundf(scale_w * sc);
            if (sc >= 32767.0f) return 32767;
            if (sc <= -32768.0f) return -32768;
            return (int32_t)sc;
        };
        std::vector<int32_t> vtab((size_t)std::max(P, 1) * VIT_WORDS, -32768);
        for (int p = 0; p < P; p++) {
            const HostProfile &h = c->prof[p];
            int32_t *T = vtab.data() + (size_t)p * VIT_WORDS + VIT_T, *E = vtab.data() + (size_t)p * VIT_WORDS + VIT_E;
            for (int k = 1; k <= h.M; k++) {
                const float *t = &h.tp[(size_t)k * 7];
                T[k * 8 + VT_BM] = wordify(logf(h.bm[k]));
                T[k * 8 + VT_MM] = wordify(logf(t[T_MM])); T[k * 8 + VT_IM] = wordify(logf(t[T_IM]));
                T[k * 8 + VT_DM] = wordify(logf(t[T_DM])); T[k * 8 + VT_MD] = wordify(logf(t[T_MD]));
                T[k * 8 + VT_DD] = wordify(logf(t[T_DD])); T[k * 8 + VT_MI] = wordify(logf(t[T_MI]));
                T[k * 8 + VT_II] = wordify(logf(t[T_II]));
                if (T[k * 8 + VT_II] == 0) T[k * 8 + VT_II] = -1;       // an II cost of 0 is not allowed in the filter
                for (int x = 0; x < 16; x++) E[x * 48 + k] = wordify(h.msc[(size_t)k * 16 + x]);
            }
        }
        CUDA_TRY(c, c->d_vtab.ensure(vtab.size() * 4));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_vtab.p, vtab.data(), vtab.size() * 4, cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
    }
    CUDA_TRY(c, c->d_mdtab.ensure(mdtab.size() * 4));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_mdtab.p, mdtab.data(), mdtab.size() * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, c->d_msvtab.ensure(msvtab.size() * 4));
    CUDA_TRY(c, c->d_etab.ensure(etab.size() * 4));
    CUDA_TRY(c, c->d_pscal.ensure(ps.size() * sizeof(ProfScalars)));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_msvtab.p, msvtab.data(), msvtab.size() * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_etab.p, etab.data(), etab.size() * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_pscal.p, ps.data(), ps.size() * sizeof(ProfScalars), cudaMemcpyHostToDevice, st));
    if (!c->d_logsum.p) {
        std::vector<float> tbl(16000);
        for (int i = 0; i < 16000; i++) tbl[i] = (float)log(1. + exp((double)-i / 1000.0));
        CUDA_TRY(c, c->d_logsum.ensure(16000 * 4));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_logsum.p, tbl.data(), 16000 * 4, cudaMemcpyHostToDevice, st));
    }
    CUDA_TRY(c, cudaStreamSynchronize(st));
    c->prof_dirty = false;
    return ITSX_OK;
}

static int ensure_lut(itsx_ctx *c)
{
    if (c->d_lut.p) return ITSX_OK;
    uint8_t lut[256];
    memset(lut, 15, sizeof(lut));
    const char *sym = "ACGTRYMKSWHBVDN";
    for (int i = 0; sym[i]; i++) {
        lut[(unsigned char)sym[i]] = (uint8_t)i;
        lut[(unsigned char)(sym[i] + 32)] = (uint8_t)i;
    }
    lut['U'] = lut['u'] = 3;
    lut['X'] = lut['x'] = 14;
    CUDA_TRY(c, c->d_lut.ensure(256));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_lut.p, lut, 256, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ITSX_OK;
}

// lengths -> word offsets -> nibble codes; per-length tables (nullsc, tjb) computed on the host
static int build_seqs(itsx_ctx *c, const uint8_t *d_ascii, const int64_t *d_off, const int32_t *d_first, int64_t nseq)
{
    cudaStream_t st = c->stream;
    int rc = ensure_lut(c);
    if (rc) return rc;
    c->nseq = nseq;
    c->pos_valid = false;
    c->stage1_done = c->stage2_done = false;
    c->Lmax = 0;
    if (nseq == 0) return ITSX_OK;
    CUDA_TRY(c, c->d_seqlen.ensure((size_t)nseq * 4));
    CUDA_TRY(c, c->d_seqwoff.ensure((size_t)(nseq + 1) * 8));
    CUDA_TRY(c, c->d_scan.ensure((size_t)(nseq + 1) * 8));
    int64_t *nw = c->d_scan.as<int64_t>();
    seqlen_kernel<<<nblk(nseq, 256), 256, 0, st>>>(d_off, d_first, nseq, c->d_seqlen.as<int32_t>(), nw);
    CUDA_TRY(c, cudaMemsetAsync(nw + nseq, 0, 8, st));
    CUDA_TRY(c, c->d_counters.ensure(64 * 8));
    int32_t *d_max = (int32_t *)(c->d_counters.as<unsigned long long>() + 40);
    int64_t *woff = c->d_seqwoff.as<int64_t>();
    int32_t *len = c->d_seqlen.as<int32_t>();
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, nw, woff, (int)nseq + 1, st); },
                        [&](void *t, size_t &b) { return cub::DeviceReduce::Max(t, b, len, d_max, (int)nseq, st); }));
    int64_t totw = 0;
    int32_t lmax = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&totw, c->d_seqwoff.as<int64_t>() + nseq, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaMemcpyAsync(&lmax, d_max, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    c->Lmax = lmax;
    CUDA_TRY(c, c->d_seqw.ensure((size_t)(totw + 8) * 4));
    seqcode_kernel<<<nblk(nseq * 32, 256), 256, 0, st>>>(d_ascii, d_off, d_first, nseq, c->d_seqwoff.as<int64_t>(),
                                                         c->d_lut.as<uint8_t>(), c->d_seqw.as<uint32_t>());
    c->launches += 4;
    // per-length tables
    std::vector<float> nullsc((size_t)lmax + 1);
    std::vector<uint8_t> tjb((size_t)lmax + 1);
    const float scale_b = (float)(3.0 / kLn2);
    for (int L = 0; L <= lmax; L++) {
        float p1 = (float)L / (float)(L + 1);
        nullsc[L] = (float)((float)L * log((double)p1) + log(1. - (double)p1));
        tjb[L] = msv_unbiased_byteify(scale_b, logf(3.0f / (float)(L + 3)));
    }
    {
        std::vector<int16_t> xw((size_t)lmax + 1);
        const float scale_w = 500.0f / (float)kLn2;
        for (int L = 0; L <= lmax; L++) {
            float sc = roundf(scale_w * logf(3.0f / ((float)L + 3.0f)));
            xw[L] = (int16_t)(sc <= -32768.0f ? -32768 : sc >= 32767.0f ? 32767 : (int)sc);
        }
        CUDA_TRY(c, c->d_xwmove.ensure(((size_t)lmax + 1) * 2));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_xwmove.p, xw.data(), xw.size() * 2, cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
    }
    CUDA_TRY(c, c->d_nullsc.ensure(((size_t)lmax + 1) * 4));
    CUDA_TRY(c, c->d_tjb.ensure((size_t)lmax + 1));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_nullsc.p, nullsc.data(), nullsc.size() * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_tjb.p, tjb.data(), tjb.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    return ITSX_OK;
}

// the search set = resident reads d_first[0..nseq); with sample ids set, every sequence is of its first read's sample
static int build_seqs_of_reads(itsx_ctx *c, const int32_t *d_first, int64_t nseq)
{
    int rc = build_seqs(c, c->d_ascii.as<uint8_t>(), c->d_off.as<int64_t>(), d_first, nseq);
    if (rc) return rc;
    if (c->have_samples && nseq > 0) {
        CUDA_TRY(c, c->d_seq_sample.ensure((size_t)nseq * 4));
        seqsample_kernel<<<nblk(nseq, 256), 256, 0, c->stream>>>(c->d_sample.as<int32_t>(), d_first, nseq,
                                                                c->d_seq_sample.as<int32_t>());
        c->launches++;
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    return ITSX_OK;
}

int search_build_seqs_from_derep(itsx_ctx *c)
{
    return build_seqs_of_reads(c, c->d_first.as<int32_t>(), c->n_unique);
}

int search_build_seqs_from_reads(itsx_ctx *c, const int32_t *d_first, int64_t nseq)
{
    c->shard_first = 0;
    c->shard_n = -1;
    return build_seqs_of_reads(c, d_first, nseq);
}

int search_build_seqs_from_host(itsx_ctx *c, const uint8_t *seq, const int64_t *off, int64_t nseq)
{
    // staged through separate buffers so that the reads of a previous itsx_derep stay resident
    static thread_local DevBuf t_ascii, t_off;
    const int64_t total = nseq ? itsx_peek_i64(off + nseq) : 0;
    CUDA_TRY(c, t_ascii.ensure((size_t)total + 64));
    CUDA_TRY(c, t_off.ensure((size_t)(nseq + 1) * 8));
    if (total) CUDA_TRY(c, cudaMemcpyAsync(t_ascii.p, seq, (size_t)total, cudaMemcpyDefault, c->stream));
    if (nseq) CUDA_TRY(c, cudaMemcpyAsync(t_off.p, off, (size_t)(nseq + 1) * 8, cudaMemcpyDefault, c->stream));
    c->shard_first = 0;
    c->shard_n = -1;
    c->have_samples = false;       // caller-supplied sequences are one sample
    c->n_samples = 1;
    return build_seqs(c, t_ascii.as<uint8_t>(), t_off.as<int64_t>(), nullptr, nseq);
}

constexpr int NLANE = 8;                   // side streams of the per-profile launches

static int ensure_lanes(itsx_ctx *c, int n)
{
    while ((int)c->lanes.size() < n) {
        cudaStream_t s;
        cudaEvent_t e;
        CUDA_TRY(c, cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        CUDA_TRY(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        c->lanes.push_back(s);
        c->lane_ev.push_back(e);
    }
    if (!c->lane_fork) CUDA_TRY(c, cudaEventCreateWithFlags(&c->lane_fork, cudaEventDisableTiming));
    return ITSX_OK;
}

// the shard of the sequence set that a search covers: sequences q0 .. q0 + qn (itsx_search_shard)
static int shard_range(itsx_ctx *c, int64_t &q0, int64_t &qn)
{
    q0 = c->shard_first;
    qn = c->shard_n < 0 ? c->nseq - q0 : c->shard_n;
    if (q0 < 0 || qn < 0 || q0 + qn > c->nseq) { c->err = "search: shard outside the sequence set"; return ITSX_EINVAL; }
    return ITSX_OK;
}

// position table, arg-max keys and the winners' multidomain flags of the shard's qn sequences; init: reset them to "no hit"
static int pos_reset(itsx_ctx *c, int64_t qn, bool init)
{
    const size_t n = (size_t)std::max<int64_t>(qn, 1);
    c->npos = qn;
    CUDA_TRY(c, c->d_pos.ensure(n * 9 * 4));
    CUDA_TRY(c, c->d_best.ensure(n * 2 * 8));
    CUDA_TRY(c, c->d_selmulti.ensure(n * 2 + 16));
    if (init && qn > 0) {
        pos_init_kernel<<<nblk(qn, 256), 256, 0, c->stream>>>(c->d_pos.as<int32_t>(), c->d_best.as<unsigned long long>(),
                                                              c->d_selmulti.as<uint8_t>(), qn);
        c->launches++;
    }
    return ITSX_OK;
}

// ---- stage 1: the filter cascade, chunk by chunk over the shard's sequences ------------------------------------------
// Events of the stage clocks.  A stage's span runs from the event that ends the stage before it to its own last event;
// the Forward stage's clock starts at S1_FILT, recorded by the bias stage or, when it runs, after the Viterbi stage.
enum { S1_CALL0, S1_MSV0, S1_MSV1, S1_FILT, S1_VIT0, S1_VIT1, S1_FB, S1_MD, S1_ENV, S1_SCORE, S1_CALL1, S1_NEV };

struct S1Call {                           // what every chunk of one search_stage1 shares
    int64_t q0 = 0, qn = 0;               // the shard
    int P = 0;
    int32_t *d_order = nullptr;           // the shard's sequences sorted by length
    unsigned long long *cnt = nullptr;    // device counters (CNT_*)
    int32_t *d_nsel = nullptr;            // survivor counts of the compactions (in d_counters)
    bool multi_sample = false;
    double lnP_certain = 0;
    Timeline<S1_NEV> tl;                  // the stages add their spans to c->sstats.ms_*
};

struct S1Chunk {                          // d_order[s0 .. s0 + ns) and its survivors
    int64_t s0 = 0;
    int ns = 0;
    int32_t n1 = 0, n2 = 0, nenv = 0;     // pairs past MSV, past bias (and Viterbi); envelopes
    std::vector<int32_t> h_bounds;        // [P + 1] per-profile slices of list2
};

// residues of the shard (cell accounting), and d_order: the shard's sequences in order of length, so that the 32 pairs
// of a warp run the same number of rows
static int s1_order(itsx_ctx *c, S1Call &s)
{
    cudaStream_t st = c->stream;
    const int64_t q0 = s.q0, qn = s.qn;
    int32_t *len = c->d_seqlen.as<int32_t>() + q0;
    long long *d_sum = (long long *)(s.cnt + 41);
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceReduce::Sum(t, b, len, d_sum, (int)qn, st); }));
    long long h = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&h, d_sum, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    double sumM = 0;
    for (auto &hp : c->prof) sumM += hp.M;
    c->sstats.msv_cells = (double)h * sumM;
    CUDA_TRY(c, c->d_order.ensure((size_t)qn * 4 * 4));
    int32_t *d_order = s.d_order = c->d_order.as<int32_t>();
    int32_t *idx_in = d_order + qn, *len_in = d_order + 2 * qn, *len_out = d_order + 3 * qn;
    iota_kernel<<<nblk(qn, 256), 256, 0, st>>>(idx_in, (int32_t)q0, qn);
    CUDA_TRY(c, cudaMemcpyAsync(len_in, len, (size_t)qn * 4, cudaMemcpyDeviceToDevice, st));
    int lbits = 1;
    while ((1 << lbits) <= c->Lmax) lbits++;
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) {
        return cub::DeviceRadixSort::SortPairs(t, b, len_in, len_out, idx_in, d_order, (int)qn, 0, lbits, st);
    }));
    c->launches += 2;
    return ITSX_OK;
}

// MSV over the chunk's pairs, then the list of the pairs that pass it (n1; its compaction is on the bias stage's clock)
static int s1_msv(itsx_ctx *c, const S1Call &s, S1Chunk &k)
{
    cudaStream_t st = c->stream;
    const size_t npair = (size_t)k.ns * s.P;
    const size_t msv_smem = (size_t)MSV_TP * MSV_TABW * 4;
    CUDA_TRY(c, cudaFuncSetAttribute(msv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msv_smem));
    CUDA_TRY(c, s.tl.record(S1_MSV0, st));
    CUDA_TRY(c, c->d_msvres.ensure(npair));
    CUDA_TRY(c, c->d_flag.ensure(npair + 16));
    dim3 grid(nblk(k.ns, MSV_THREADS), (s.P + MSV_TP - 1) / MSV_TP);
    msv_kernel<<<grid, MSV_THREADS, msv_smem, st>>>(c->d_seqw.as<uint32_t>(), c->d_seqwoff.as<int64_t>(),
                                                    c->d_seqlen.as<int32_t>(), s.d_order, k.s0, k.ns, c->d_msvtab.as<uint32_t>(),
                                                    c->d_pscal.as<ProfScalars>(), s.P, c->d_tjb.as<uint8_t>(),
                                                    c->d_nullsc.as<float>(), c->prm.F1,
                                                    c->d_msvres.as<uint8_t>(), c->d_flag.as<uint8_t>());
    c->launches++;
    CUDA_TRY(c, s.tl.record(S1_MSV1, st));
    CUDA_TRY(c, c->d_list.ensure(npair * 4 + 16));
    cub::CountingInputIterator<int32_t> iota(0);
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) {
        return cub::DeviceSelect::Flagged(t, b, iota, c->d_flag.as<uint8_t>(), c->d_list.as<int32_t>(), s.d_nsel, (int)npair, st);
    }));
    CUDA_TRY(c, cudaMemcpyAsync(&k.n1, s.d_nsel, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    c->sstats.n_past_msv += k.n1;
    c->sstats.ms_msv += s.tl.ms(S1_MSV0, S1_MSV1);
    return ITSX_OK;
}

// entries of (list, sc) whose flag is set, in order, to (list_out, sc_out); *d_n receives their number
static cudaError_t compact_list_sc(itsx_ctx *c, int32_t *list, float *sc, uint8_t *flag, int32_t *list_out, float *sc_out,
                                   int32_t *d_n, int n)
{
    cudaStream_t st = c->stream;
    return cub_run(c, [&](void *t, size_t &b) { return cub::DeviceSelect::Flagged(t, b, list, flag, list_out, d_n, n, st); },
                   [&](void *t, size_t &b) { return cub::DeviceSelect::Flagged(t, b, sc, flag, sc_out, d_n, n, st); });
}

// bias filter over the n1 MSV survivors: list2 / fsc2 hold the n2 that pass, h_bounds their per-profile slices
static int s1_bias(itsx_ctx *c, const S1Call &s, S1Chunk &k)
{
    cudaStream_t st = c->stream;
    const int P = s.P, n1 = k.n1;
    CUDA_TRY(c, c->d_filtersc.ensure((size_t)n1 * 4));
    CUDA_TRY(c, c->d_ndom.ensure((size_t)n1 + 16));   // reused as flag2 here
    bias_kernel<<<nblk(n1, 128), 128, 0, st>>>(c->d_list.as<int32_t>(), s.d_nsel, s.d_order, k.s0, k.ns, c->d_seqw.as<uint32_t>(),
                                               c->d_seqwoff.as<int64_t>(), c->d_seqlen.as<int32_t>(),
                                               c->d_pscal.as<ProfScalars>(), c->d_msvres.as<uint8_t>(),
                                               c->d_tjb.as<uint8_t>(), c->prm.F1, c->prm.F2, c->d_filtersc.as<float>(),
                                               c->d_ndom.as<uint8_t>(), s.cnt);
    CUDA_TRY(c, c->d_list2.ensure((size_t)n1 * 4 + 16));
    CUDA_TRY(c, c->d_fsc2.ensure((size_t)n1 * 4 + 16));
    int32_t *d_nsel2 = s.d_nsel + 1;
    CUDA_TRY(c, compact_list_sc(c, c->d_list.as<int32_t>(), c->d_filtersc.as<float>(), c->d_ndom.as<uint8_t>(),
                                c->d_list2.as<int32_t>(), c->d_fsc2.as<float>(), d_nsel2, n1));
    CUDA_TRY(c, c->d_bounds.ensure((size_t)(P + 1) * 8));
    bounds_kernel<<<nblk(P + 1, 128), 128, 0, st>>>(c->d_list2.as<int32_t>(), d_nsel2, k.ns, P, c->d_bounds.as<int32_t>());
    c->launches += 2;
    k.h_bounds.resize((size_t)P + 1);
    CUDA_TRY(c, cudaMemcpyAsync(&k.n2, d_nsel2, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaMemcpyAsync(k.h_bounds.data(), c->d_bounds.p, (size_t)(P + 1) * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, s.tl.record(S1_FILT, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    c->sstats.n_past_bias += k.n2;
    c->sstats.ms_bias += s.tl.ms(S1_MSV1, S1_FILT);
    return ITSX_OK;
}

// Viterbi filter for the entries with F2 < P(MSV + bias) <= F1 (never under the reference's F1 == F2): list2 / fsc2 and
// h_bounds keep the n2 entries that pass it
static int s1_viterbi(itsx_ctx *c, const S1Call &s, S1Chunk &k)
{
    cudaStream_t st = c->stream;
    const int P = s.P, n1 = k.n1, n2 = k.n2;
    CUDA_TRY(c, s.tl.record(S1_VIT0, st));
    // the "needs the filter" marks of the surviving entries, compacted like the list itself
    CUDA_TRY(c, c->d_vneed.ensure((size_t)n1 + 16));
    CUDA_TRY(c, c->d_vpass.ensure((size_t)n2 + 16));
    int32_t *d_nsel3 = s.d_nsel + 2;
    uint8_t *d_run = c->d_ndom.as<uint8_t>();      // the bias flags; once consumed, the "run" marks
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) {
        return cub::DeviceSelect::Flagged(t, b, d_run, d_run, c->d_vneed.as<uint8_t>(), d_nsel3, n1, st);
    }));
    // worklist of the entries the filter has to look at (full warps), its per-profile slices
    CUDA_TRY(c, c->d_list.ensure((size_t)n2 * 4 * 2 + 64));
    vneed_flag_kernel<<<nblk(n2, 256), 256, 0, st>>>(c->d_vneed.as<uint8_t>(), n2, d_run, c->d_vpass.as<uint8_t>());
    int32_t *d_vidx = c->d_list.as<int32_t>() + n2;         // second half of d_list (first half: compaction output below)
    int32_t *d_nv = s.d_nsel + 3;
    cub::CountingInputIterator<int32_t> iota0(0);
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceSelect::Flagged(t, b, iota0, d_run, d_vidx, d_nv, n2, st); }));
    vbounds_kernel<<<nblk(P + 1, 128), 128, 0, st>>>(c->d_list2.as<int32_t>(), d_vidx, d_nv, k.ns, P,
                                                     c->d_bounds.as<int32_t>() + (P + 1));
    std::vector<int32_t> h_vb((size_t)P + 1);
    CUDA_TRY(c, cudaMemcpyAsync(h_vb.data(), c->d_bounds.as<int32_t>() + (P + 1), (size_t)(P + 1) * 4,
                                cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    c->launches += 3;
    CUDA_TRY(c, fork_lanes(c, NLANE));
    int vrr = 0;
    for (int p = 0; p < P; p++) {
        const int b0 = h_vb[p], cntp = h_vb[p + 1] - b0;
        if (cntp <= 0) continue;
        VitArgs va;
        va.list = c->d_list2.as<int32_t>(); va.filtersc = c->d_fsc2.as<float>();
        va.vidx = d_vidx + b0; va.count = cntp;
        va.order = s.d_order; va.s0 = k.s0; va.ns = k.ns; va.prof = p;
        va.seqw = c->d_seqw.as<uint32_t>(); va.woff = c->d_seqwoff.as<int64_t>(); va.seqlen = c->d_seqlen.as<int32_t>();
        va.vtab = c->d_vtab.as<int32_t>() + (size_t)p * VIT_WORDS;
        va.xwmove = c->d_xwmove.as<int16_t>();
        va.xw_E = (int)roundf(500.0f / (float)kLn2 * (-(float)kLn2));
        va.vmu = c->prof[p].ev[EV_VMU]; va.vlambda = c->prof[p].ev[EV_VLAMBDA];
        va.F2 = c->prm.F2;
        va.pass = c->d_vpass.as<uint8_t>();
        va.counters = s.cnt;
        vit_kernel<<<nblk(cntp, 128), 128, 0, c->lanes[vrr++ % NLANE]>>>(va);
        c->launches++;
    }
    CUDA_TRY(c, join_lanes(c, NLANE));
    // survivors: list2 / fsc2 compacted by the pass flags (through the bias stage's buffers, then back)
    CUDA_TRY(c, compact_list_sc(c, c->d_list2.as<int32_t>(), c->d_fsc2.as<float>(), c->d_vpass.as<uint8_t>(),
                                c->d_list.as<int32_t>(), c->d_filtersc.as<float>(), d_nsel3, n2));
    int32_t n3 = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&n3, d_nsel3, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    if (n3 > 0) {
        CUDA_TRY(c, cudaMemcpyAsync(c->d_list2.p, c->d_list.p, (size_t)n3 * 4, cudaMemcpyDeviceToDevice, st));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_fsc2.p, c->d_filtersc.p, (size_t)n3 * 4, cudaMemcpyDeviceToDevice, st));
    }
    bounds_kernel<<<nblk(P + 1, 128), 128, 0, st>>>(c->d_list2.as<int32_t>(), d_nsel3, k.ns, P, c->d_bounds.as<int32_t>());
    c->launches += 3;
    CUDA_TRY(c, cudaMemcpyAsync(k.h_bounds.data(), c->d_bounds.p, (size_t)(P + 1) * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, s.tl.record(S1_VIT1, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    c->sstats.ms_vit += s.tl.ms(S1_VIT0, S1_VIT1);
    k.n2 = n3;
    CUDA_TRY(c, s.tl.record(S1_FILT, st));
    return ITSX_OK;
}

// Forward / Backward / posterior decoding of the n2 entries: one launch per profile (in pieces) over the side streams
static int s1_fwdbck(itsx_ctx *c, const S1Call &s, const S1Chunk &k)
{
    const int n2 = k.n2, Lmax = c->Lmax;
    CUDA_TRY(c, c->d_fwdsc.ensure((size_t)n2 * 4));
    CUDA_TRY(c, c->d_pairout.ensure((size_t)n2 * 4));
    CUDA_TRY(c, c->d_ndom.ensure((size_t)n2 + 16));
    CUDA_TRY(c, c->d_env.ensure((size_t)n2 * ITSX_MAXDOM * 2 * 4));
    const size_t slab = (size_t)(Lmax + 1) * SPEC_C * 32 * 4;
    // the slab of a launch holds all its tiles (fbdec_kernel reads them back): a profile's worklist goes in pieces of
    // at most two tiles per resident warp, and no more than fit the scratch budget
    const int fb_warps_per_lane = c->sm_count * FB_CTAS_PER_SM * (FB_THREADS / 32);
    const int fb_piece_tiles = (int)std::max<size_t>(
        1, std::min<size_t>((size_t)fb_warps_per_lane * 2, FB_SCRATCH_BUDGET / (slab * NLANE)));
    CUDA_TRY(c, c->d_spec.ensure(slab * (size_t)fb_piece_tiles * NLANE));
    CUDA_TRY(c, c->d_fbscale.ensure((size_t)n2 * 4));
    CUDA_TRY(c, fork_lanes(c, NLANE));
    int lane_rr = 0;
    for (int p = 0; p < s.P; p++) {
        const int b0 = k.h_bounds[p], cntp = k.h_bounds[p + 1] - b0;
        if (cntp <= 0) continue;
        const int l = lane_rr++ % NLANE;
        FbArgs fa;
        fa.order = s.d_order; fa.s0 = k.s0; fa.ns = k.ns; fa.prof = p;
        fa.seqw = c->d_seqw.as<uint32_t>(); fa.woff = c->d_seqwoff.as<int64_t>(); fa.seqlen = c->d_seqlen.as<int32_t>();
        fa.etab = c->d_etab.as<float>() + (size_t)p * (MAXM + 1) * 16;
        fa.Lmax = Lmax;
        fa.tau = c->prof[p].ev[EV_FTAU]; fa.lambda = c->prof[p].ev[EV_FLAMBDA];
        fa.F3 = c->prm.F3;
        fa.e_move = expf(-(float)kLn2);
        fa.counters = s.cnt;
        const int wpc = FB_THREADS / 32;
        fa.spec = (float *)(c->d_spec.as<char>() + slab * (size_t)fb_piece_tiles * l);
        for (int e0 = 0; e0 < cntp; e0 += fb_piece_tiles * 32) {
            FbArgs fp = fa;
            const int o = b0 + e0;          // the piece: entries o .. o + count of list2
            fp.count = std::min(cntp - e0, fb_piece_tiles * 32);
            fp.list = c->d_list2.as<int32_t>() + o; fp.filtersc = c->d_fsc2.as<float>() + o;
            fp.fwdsc = c->d_fwdsc.as<float>() + o; fp.bcksc = c->d_pairout.as<float>() + o;
            fp.ndom = c->d_ndom.as<uint8_t>() + o; fp.env = c->d_env.as<int32_t>() + (size_t)o * ITSX_MAXDOM * 2;
            fp.scale = c->d_fbscale.as<float>() + o;
            const int tiles = (fp.count + 31) / 32;
            const int ctas = std::min((tiles + wpc - 1) / wpc, c->sm_count * FB_CTAS_PER_SM);
            fb_kernel<<<ctas, FB_THREADS, 0, c->lanes[l]>>>(c->pconst[p], fp);
            fbdec_kernel<<<(tiles + 3) / 4, 128, 0, c->lanes[l]>>>(fp);
            c->launches += 2;
        }
    }
    CUDA_TRY(c, join_lanes(c, NLANE));
    CUDA_TRY(c, s.tl.record(S1_FB, c->stream));
    return ITSX_OK;
}

// multidomain regions: stochastic-traceback clustering replaces the region by its cluster envelopes
static int s1_multidomain(itsx_ctx *c, const S1Call &s, const S1Chunk &k)
{
    cudaStream_t st = c->stream;
    const int n2 = k.n2;
    CUDA_TRY(c, c->d_envdc.ensure((size_t)n2 * ITSX_MAXDOM * 4));
    CUDA_TRY(c, c->d_n2reg.ensure((size_t)n2 * 4));
    CUDA_TRY(c, cudaMemsetAsync(c->d_n2reg.p, 0, (size_t)n2 * 4, st));
    // flagged regions per entry -> prefix sum -> region list in entry order
    int32_t h_nregions = 0, *d_base = nullptr;
    if (c->prm.resolve_multidomain) {
        CUDA_TRY(c, c->d_mdlist.ensure((size_t)(n2 + 1) * 2 * 4));
        int32_t *d_nreg = c->d_mdlist.as<int32_t>();
        d_base = d_nreg + (n2 + 1);
        mdcount_kernel<<<nblk(n2 + 1, 256), 256, 0, st>>>(c->d_ndom.as<uint8_t>(), c->d_env.as<int32_t>(), n2, d_nreg);
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, d_nreg, d_base, n2 + 1, st); }));
        c->launches += 2;
        CUDA_TRY(c, cudaMemcpyAsync(&h_nregions, d_base + n2, 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
    }
    if (h_nregions > 0) {
        const int NR = h_nregions;
        CUDA_TRY(c, c->d_mdreg.ensure(((size_t)NR * 3 + (size_t)(NR + 1) * 2) * 4));
        int32_t *reg_ent = c->d_mdreg.as<int32_t>(), *reg_i = reg_ent + NR, *reg_j = reg_i + NR,
                *reg_rows = reg_j + NR, *reg_row = reg_rows + (NR + 1);
        CUDA_TRY(c, cudaMemsetAsync(reg_rows + NR, 0, 4, st));
        mdregs_kernel<<<nblk(n2, 256), 256, 0, st>>>(c->d_ndom.as<uint8_t>(), c->d_env.as<int32_t>(), n2, d_base,
                                                    reg_ent, reg_i, reg_j, reg_rows);
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, reg_rows, reg_row, NR + 1, st); }));
        c->launches += 2;
        std::vector<int32_t> h_row((size_t)NR + 1);
        CUDA_TRY(c, cudaMemcpyAsync(h_row.data(), reg_row, (size_t)(NR + 1) * 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        CUDA_TRY(c, c->d_mdres.ensure((size_t)NR * sizeof(MdRes)));
        MdStreams streams;
        const uint32_t x0 = md_rng_state0(42u);
        for (int t = 0; t < MD_NSAMPLES; t++) streams.x[t] = md_rng_jump(x0, (uint64_t)t << MD_STREAM_LOG2);
        MdArgs ma;
        ma.reg_ent = reg_ent; ma.reg_i = reg_i; ma.reg_j = reg_j; ma.reg_row = reg_row;
        ma.list = c->d_list2.as<int32_t>(); ma.order = s.d_order; ma.s0 = k.s0; ma.ns = k.ns;
        ma.seqw = c->d_seqw.as<uint32_t>(); ma.woff = c->d_seqwoff.as<int64_t>(); ma.seqlen = c->d_seqlen.as<int32_t>();
        ma.mdtab = c->d_mdtab.as<float>(); ma.etab = c->d_etab.as<float>(); ma.pscal = c->d_pscal.as<ProfScalars>();
        ma.res = c->d_mdres.as<MdRes>();
        ma.e_move = expf(-(float)kLn2);
        ma.counters = s.cnt;
        // chunks of regions: slabs (matrix + row tables) and trace records within a fixed HBM budget; consecutive
        // chunks alternate between two side streams with their own buffers, so that the latency-bound Forward fill of
        // one chunk runs under the issue-bound tracebacks / clustering of the other
        const size_t row_bytes = (size_t)MD_W * 16 + sizeof(MdRow), reg_bytes = (size_t)MD_TRACE_BYTES;
        const size_t budget = (size_t)3 << 30;
        struct MdChunk { int r0, r1, maxrows, ctas; size_t rows; };
        std::vector<MdChunk> chunks;
        const size_t cl_smem = sizeof(MdClustSmem) * MDC_WARPS;
        CUDA_TRY(c, cudaFuncSetAttribute(mdclust_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cl_smem));
        int cl_per_sm = 0;      // resident CTAs per SM at this shared-memory size: the grid is ONE wave
        CUDA_TRY(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cl_per_sm, mdclust_kernel, MDC_WARPS * 32, cl_smem));
        size_t need_cell[2] = {0, 0}, need_trace[2] = {0, 0}, need_scr[2] = {0, 0};
        for (int r0 = 0; r0 < NR;) {
            int r1 = r0 + 1;
            while (r1 < NR && (size_t)(h_row[r1 + 1] - h_row[r0]) * row_bytes + (size_t)(r1 + 1 - r0) * reg_bytes <= budget)
                r1++;
            MdChunk ch;
            ch.r0 = r0; ch.r1 = r1; ch.rows = (size_t)(h_row[r1] - h_row[r0]); ch.maxrows = 0;
            for (int r = r0; r < r1; r++) ch.maxrows = std::max(ch.maxrows, h_row[r + 1] - h_row[r]);
            ch.ctas = std::min((r1 - r0 + MDC_WARPS - 1) / MDC_WARPS, c->sm_count * std::max(cl_per_sm, 1));
            const int par = (int)(chunks.size() & 1);
            need_cell[par] = std::max(need_cell[par], ch.rows * row_bytes);
            need_trace[par] = std::max(need_trace[par], (size_t)(r1 - r0) * reg_bytes);
            need_scr[par] = std::max(need_scr[par], md_clust_bytes(ch.maxrows) * (size_t)ch.ctas * MDC_WARPS);
            chunks.push_back(ch);
            r0 = r1;
        }
        for (int par = 0; par < 2; par++) {
            CUDA_TRY(c, c->d_mdcell[par].ensure(need_cell[par]));
            CUDA_TRY(c, c->d_mdtrace[par].ensure(need_trace[par]));
            CUDA_TRY(c, c->d_mdscratch[par].ensure(need_scr[par]));
        }
        CUDA_TRY(c, fork_lanes(c, 2));
        for (size_t ci = 0; ci < chunks.size(); ci++) {
            const MdChunk &ch = chunks[ci];
            const int par = (int)(ci & 1);
            cudaStream_t ms = c->lanes[par];
            ma.r0 = ch.r0; ma.r1 = ch.r1; ma.row0 = h_row[ch.r0];
            ma.cell = c->d_mdcell[par].as<float4>();
            ma.rowrec = (MdRow *)(c->d_mdcell[par].as<char>() + ch.rows * MD_W * 16);
            ma.trace = c->d_mdtrace[par].as<char>();
            ma.maxrows = ch.maxrows;
            ma.per_thread = md_clust_bytes(ch.maxrows);
            ma.scratch = c->d_mdscratch[par].as<char>();
            mdfwd_kernel<<<nblk(ch.r1 - ch.r0, 64), 64, 0, ms>>>(ma);
            mdtrace_kernel<<<nblk((int64_t)(ch.r1 - ch.r0) * MD_NSAMPLES, 128), 128, 0, ms>>>(ma, streams);
            mdclust_kernel<<<ch.ctas, MDC_WARPS * 32, cl_smem, ms>>>(ma);
            c->launches += 3;
        }
        CUDA_TRY(c, join_lanes(c, 2));
        mdapply_kernel<<<nblk(n2, 256), 256, 0, st>>>(c->d_ndom.as<uint8_t>(), c->d_env.as<int32_t>(), n2, d_base,
                                                     c->d_mdres.as<MdRes>(), c->d_envdc.as<float>(),
                                                     c->d_n2reg.as<float>(), s.cnt);
        c->launches++;
    }
    CUDA_TRY(c, s.tl.record(S1_MD, st));
    return ITSX_OK;
}

// envelope worklist (sorted by profile and envelope length) and unihit rescoring of every envelope (nenv)
static int s1_envelopes(itsx_ctx *c, const S1Call &s, S1Chunk &k)
{
    cudaStream_t st = c->stream;
    const int P = s.P, n2 = k.n2;
    CUDA_TRY(c, c->d_scan.ensure((size_t)(n2 + 1) * 4));
    CUDA_TRY(c, c->d_envoff.ensure((size_t)(n2 + 1) * 4));
    ndom_widen_kernel<<<nblk(n2 + 1, 256), 256, 0, st>>>(c->d_ndom.as<uint8_t>(), n2, c->d_scan.as<int32_t>());
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) {
        return cub::DeviceScan::ExclusiveSum(t, b, c->d_scan.as<int32_t>(), c->d_envoff.as<int32_t>(), n2 + 1, st);
    }));
    gather_bounds_kernel<<<nblk(P + 1, 128), 128, 0, st>>>(c->d_envoff.as<int32_t>(), c->d_bounds.as<int32_t>(), P,
                                                           c->d_bounds.as<int32_t>() + (P + 1));
    c->launches += 2;
    std::vector<int32_t> h_envb((size_t)P + 1);
    CUDA_TRY(c, cudaMemcpyAsync(h_envb.data(), c->d_bounds.as<int32_t>() + (P + 1), (size_t)(P + 1) * 4,
                                cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    const int nenv = k.nenv = h_envb[P];
    if (nenv > 0) {
        CUDA_TRY(c, c->d_envout.ensure((size_t)nenv * 20 * 4));
        // worklist sorted by (profile, envelope length): two ping-pong buffers for the radix sort
        CUDA_TRY(c, c->d_envwork.ensure((size_t)nenv * 4 * 4));
        int32_t *wk_in = c->d_envwork.as<int32_t>(), *wk_out = wk_in + nenv;
        uint32_t *key_in = (uint32_t *)(wk_in + 2 * (size_t)nenv), *key_out = key_in + nenv;
        envwork_kernel<<<nblk(n2, 256), 256, 0, st>>>(c->d_ndom.as<uint8_t>(), c->d_envoff.as<int32_t>(), n2,
                                                      c->d_list2.as<int32_t>(), k.ns, c->d_env.as<int32_t>(), wk_in,
                                                      key_in);
        int pbits = 1;
        while ((1 << pbits) < P) pbits++;
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) {
            return cub::DeviceRadixSort::SortPairs(t, b, key_in, key_out, wk_in, wk_out, nenv, 0, 12 + pbits, st);
        }));
        c->launches += 2;
        // envelopes are at most Lmax long; scratch per warp of the grid, whose size the budget bounds
        const size_t eslab = (size_t)(c->Lmax + 1) * ENV_ROWF * 32 * 4;
        const int env_wpc = ENV_THREADS / 32;
        const int env_warps = (int)std::max<size_t>(
            env_wpc, std::min<size_t>(c->sm_count * ENV_CTAS_PER_SM * env_wpc,
                                      ENV_SCRATCH_BUDGET / (eslab * NLANE) / env_wpc * env_wpc));
        const size_t env_smem = (size_t)(ENV_THREADS / 32) * ENV_RING * (ENV_ROWBYTES + 8);
        CUDA_TRY(c, cudaFuncSetAttribute(env_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)env_smem));
        CUDA_TRY(c, c->d_envscratch.ensure(eslab * env_warps * NLANE));
        CUDA_TRY(c, fork_lanes(c, NLANE));
        int lane_rr = 0;
        for (int p = 0; p < P; p++) {
            const int e0 = h_envb[p], cnte = h_envb[p + 1] - e0;
            if (cnte <= 0) continue;
            const int l = lane_rr++ % NLANE;
            EnvArgs ea;
            ea.work = wk_out + e0;
            ea.envoff = c->d_envoff.as<int32_t>();
            ea.count = cnte;
            ea.list = c->d_list2.as<int32_t>();
            ea.env = c->d_env.as<int32_t>();
            ea.order = s.d_order; ea.s0 = k.s0; ea.ns = k.ns; ea.prof = p;
            ea.seqw = c->d_seqw.as<uint32_t>(); ea.woff = c->d_seqwoff.as<int64_t>(); ea.seqlen = c->d_seqlen.as<int32_t>();
            ea.etab = c->d_etab.as<float>() + (size_t)p * (MAXM + 1) * 16;
            ea.scratch = (float *)(c->d_envscratch.as<char>() + eslab * env_warps * l);
            ea.Ldmax = c->Lmax;
            ea.out = c->d_envout.as<float>();
            ea.out_base = e0;
            ea.counters = s.cnt;
            const int tiles = (cnte + 31) / 32;
            const int ctas = std::min((tiles + env_wpc - 1) / env_wpc, env_warps / env_wpc);
            env_kernel<<<ctas, ENV_THREADS, env_smem, c->lanes[l]>>>(c->pconst[p], ea);
            c->launches++;
        }
        CUDA_TRY(c, join_lanes(c, NLANE));
    }
    CUDA_TRY(c, s.tl.record(S1_ENV, st));
    return ITSX_OK;
}

// sequence and domain scores of the chunk's envelopes; in compact mode (keep_rows 2) the per-sequence selection too.
// The chunk's work ends here: the Forward, resolver, envelope and score spans are read after its synchronisation.
static int s1_scores(itsx_ctx *c, const S1Call &s, const S1Chunk &k)
{
    cudaStream_t st = c->stream;
    itsx_search_stats &ss = c->sstats;
    if (k.nenv > 0) {
        CUDA_TRY(c, c->d_doms.ensure((size_t)(c->ndom + k.nenv) * sizeof(DomRec), true, st));
        FinalArgs fa;
        fa.list = c->d_list2.as<int32_t>(); fa.n = k.n2; fa.order = s.d_order; fa.s0 = k.s0; fa.ns = k.ns;
        fa.seqw = c->d_seqw.as<uint32_t>(); fa.woff = c->d_seqwoff.as<int64_t>(); fa.seqlen = c->d_seqlen.as<int32_t>();
        fa.pscal = c->d_pscal.as<ProfScalars>(); fa.nullsctab = c->d_nullsc.as<float>();
        fa.logsum = c->d_logsum.as<float>(); fa.fwdsc = c->d_fwdsc.as<float>();
        fa.ndom = c->d_ndom.as<uint8_t>(); fa.envoff = c->d_envoff.as<int32_t>(); fa.env = c->d_env.as<int32_t>();
        fa.envdc = c->d_envdc.as<float>(); fa.n2reg = c->d_n2reg.as<float>();
        fa.envout = c->d_envout.as<float>(); fa.T = c->prm.T;
        fa.doms = c->d_doms.as<DomRec>() + (c->compact ? 0 : c->ndom);
        fa.nrep = c->d_nrep.as<int32_t>(); fa.counters = s.cnt;
        fa.seq_sample = s.multi_sample ? c->d_seq_sample.as<int32_t>() : nullptr; fa.P = s.P;
        fa.compact = c->compact ? 1 : 0;
        fa.best = c->d_best.as<unsigned long long>(); fa.nseq = s.qn; fa.seq_first = s.q0;
        fa.lnP_certain = s.lnP_certain;
        final_kernel<<<nblk(k.n2, 128), 128, 0, st>>>(fa);
        c->launches++;
        ss.n_domains += k.nenv;
        if (c->compact) {
            compact_select_kernel<<<nblk(k.n2, 128), 128, 0, st>>>(fa, s.cnt + CNT_NDOM, c->d_pos.as<int32_t>(),
                                                                  c->d_selmulti.as<uint8_t>());
            c->launches++;
            unsigned long long cur = 0;
            CUDA_TRY(c, cudaMemcpyAsync(&cur, s.cnt + CNT_NDOM, 8, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(c, cudaStreamSynchronize(st));
            c->ndom = (int64_t)cur;
        } else {
            c->ndom += k.nenv;
        }
    }
    CUDA_TRY(c, s.tl.record(S1_SCORE, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    ss.ms_fwd += s.tl.ms(S1_FILT, S1_FB);
    ss.ms_mdom += s.tl.ms(S1_FB, S1_MD);
    ss.ms_env += s.tl.ms(S1_MD, S1_ENV);
    ss.ms_final += s.tl.ms(S1_ENV, S1_SCORE);
    return ITSX_OK;
}

int search_stage1(itsx_ctx *c)
{
    cudaStream_t st = c->stream;
    int rc = search_upload_profiles(c);
    if (rc) return rc;
    S1Call s;
    const int P = s.P = (int)c->prof.size();
    itsx_search_stats &ss = c->sstats;
    ss = itsx_search_stats{};
    c->ndom = 0;
    c->stage1_done = c->stage2_done = false;
    c->pos_valid = false;
    if ((rc = shard_range(c, s.q0, s.qn))) return rc;
    const int64_t qn = s.qn;
    ss.n_seq = qn; ss.n_prof = P; ss.n_pairs = qn * P;
    CUDA_TRY(c, c->d_counters.ensure(64 * 8));
    CUDA_TRY(c, cudaMemsetAsync(c->d_counters.p, 0, 32 * 8, st));
    s.multi_sample = c->have_samples && c->n_samples > 1 && c->d_seq_sample.p != nullptr;
    const size_t nrep_n = (size_t)P * (s.multi_sample ? c->n_samples : 1);
    CUDA_TRY(c, c->d_nrep.ensure(std::max<size_t>(nrep_n, 1) * 4));
    CUDA_TRY(c, cudaMemsetAsync(c->d_nrep.p, 0, std::max<size_t>(nrep_n, 1) * 4, st));
    c->h_nrep.assign(nrep_n, 0);
    c->compact = false;
    c->stage2_applied = false;
    c->n_certain_rows = 0;
    if (P == 0 || qn == 0) { c->stage1_done = true; return ITSX_OK; }
    c->compact = c->prm.keep_rows == 2 || (c->prm.keep_rows == 0 && qn > 200000);
    // position table, arg-max keys and the winners' multidomain flags live from stage 1 on (compact mode fills them as
    // it goes; mode 1 re-initialises them in stage 2, which may then be repeated with another domZ)
    if ((rc = pos_reset(c, qn, true))) return rc;
    const double domz_upper = c->prm.domz_upper > 0 ? (double)c->prm.domz_upper : (double)qn;
    s.lnP_certain = log(c->prm.domE / std::max(domz_upper, 1.0));
    if ((rc = ensure_lanes(c, NLANE))) return rc;
    s.cnt = c->d_counters.as<unsigned long long>();
    s.d_nsel = (int32_t *)(s.cnt + 42);
    CUDA_TRY(c, s.tl.status);
    CUDA_TRY(c, s.tl.record(S1_CALL0, st));
    if ((rc = s1_order(c, s))) return rc;

    // a chunk's scratch grows with its survivors (up to ~half of the pairs on amplicons: 64 B of envelope list + ~110 B
    // of rescoring output each), so chunks are capped at 2^27 pairs (~12 GB of scratch at 45 % survival)
    int64_t chunk = std::min<int64_t>(qn, std::max<int64_t>(1024, (1LL << 27) / P));
    chunk = std::min<int64_t>(chunk, 1LL << 22);
    for (int64_t s0 = 0; s0 < qn; s0 += chunk) {          // s0: offset into d_order
        S1Chunk k{s0, (int)std::min<int64_t>(chunk, qn - s0)};
        if ((rc = s1_msv(c, s, k))) return rc;
        if (k.n1 == 0) continue;
        if ((rc = s1_bias(c, s, k))) return rc;
        if (k.n2 == 0) continue;
        if (c->prm.F2 < c->prm.F1 && (rc = s1_viterbi(c, s, k))) return rc;
        ss.n_past_vit += k.n2;
        if (k.n2 == 0) continue;
        if ((rc = s1_fwdbck(c, s, k)) || (rc = s1_multidomain(c, s, k)) || (rc = s1_envelopes(c, s, k)) ||
            (rc = s1_scores(c, s, k)))
            return rc;
    }

    CUDA_TRY(c, s.tl.record(S1_CALL1, st));
    unsigned long long h_cnt[CNT_N];
    CUDA_TRY(c, cudaMemcpyAsync(h_cnt, s.cnt, sizeof(h_cnt), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->h_nrep.data(), c->d_nrep.p, nrep_n * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    ss.n_past_fwd = (int64_t)h_cnt[CNT_PAST_FWD];
    ss.n_hits_reported = (int64_t)h_cnt[CNT_HITS_REPORTED];
    c->n_certain_rows = (int64_t)h_cnt[CNT_CERTAIN];
    ss.n_multidomain_regions = (int64_t)h_cnt[CNT_MULTI];
    ss.n_dom_overflow = (int64_t)h_cnt[CNT_DOM_OVERFLOW];
    ss.bias_rows = (double)h_cnt[CNT_BIAS_ROWS];
    ss.vit_cells = (double)h_cnt[CNT_VIT_ROWS] * MAXM;
    ss.n_vit_run = (int64_t)h_cnt[CNT_VIT_RUN];
    ss.fwd_cells = (double)h_cnt[CNT_FWD_ROWS] * MAXM;
    ss.bck_cells = (double)h_cnt[CNT_BCK_ROWS] * MAXM;
    ss.env_cells = (double)h_cnt[CNT_ENV_ROWS] * MAXM * 2;
    ss.ms_total = s.tl.ms(S1_CALL0, S1_CALL1);
    c->stage1_done = true;
    if (ss.n_dom_overflow > 0) {
        c->err = "search: a hit had more than ITSX_MAXDOM envelopes";
        return ITSX_ELIMIT;
    }
    return ITSX_OK;
}

int search_stage2(itsx_ctx *c)
{
    if (!c->stage1_done) { c->err = "search: stage2 before stage1"; return ITSX_EINVAL; }
    cudaStream_t st = c->stream;
    const int P = (int)c->prof.size();
    // itsx_profiles_set_sides after stage1 (ItsPosition learns the region only now): refresh the tables
    int rc = search_upload_profiles(c);
    if (rc) return rc;
    int64_t q0, qn;
    if ((rc = shard_range(c, q0, qn))) return rc;
    if (c->compact && c->stage2_applied) {
        c->err = "search: stage 2 was already applied to this compact search (keep_rows 2); run stage 1 again";
        return ITSX_EINVAL;
    }
    Timeline<2> tl;
    CUDA_TRY(c, tl.status);
    CUDA_TRY(c, tl.record(0, st));
    if ((rc = pos_reset(c, qn, !c->compact))) return rc;
    unsigned long long *cnt = c->d_counters.as<unsigned long long>();
    c->sstats.n_domains_reported = c->compact ? c->n_certain_rows : 0;
    c->sstats.n_selected_multidomain = 0;
    if (qn > 0 && P > 0) {
        CUDA_TRY(c, cudaMemsetAsync(cnt + CNT_DOM_REPORTED, 0, 8, st));
        CUDA_TRY(c, cudaMemsetAsync(cnt + CNT_SEL_MULTI, 0, 8, st));
        if (c->ndom > 0) {
            const bool multi_sample = c->have_samples && c->n_samples > 1 && c->h_nrep.size() == (size_t)P * c->n_samples;
            CUDA_TRY(c, cudaMemcpyAsync(c->d_nrep.p, c->h_nrep.data(), c->h_nrep.size() * 4, cudaMemcpyHostToDevice, st));
            select_kernel<<<nblk(c->ndom, 256), 256, 0, st>>>(c->d_doms.as<DomRec>(), c->ndom, c->d_nrep.as<int32_t>(),
                                                              multi_sample ? c->d_seq_sample.as<int32_t>() : nullptr, P,
                                                              c->d_pscal.as<ProfScalars>(), c->prm.domE,
                                                              c->d_best.as<unsigned long long>(), qn, q0, cnt);
            best_kernel<<<nblk(c->ndom, 256), 256, 0, st>>>(c->d_doms.as<DomRec>(), c->ndom, c->d_pscal.as<ProfScalars>(),
                                                            c->d_best.as<unsigned long long>(), qn, q0,
                                                            c->d_pos.as<int32_t>(), c->d_selmulti.as<uint8_t>());
            c->launches += 2;
        }
        selmulti_count_kernel<<<nblk(2 * qn, 256), 256, 0, st>>>(c->d_selmulti.as<uint8_t>(), 2 * qn, cnt);
        c->launches++;
        unsigned long long nr = 0, nsm = 0;
        CUDA_TRY(c, cudaMemcpyAsync(&nr, cnt + CNT_DOM_REPORTED, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaMemcpyAsync(&nsm, cnt + CNT_SEL_MULTI, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        c->sstats.n_domains_reported += (int64_t)nr;
        c->sstats.n_selected_multidomain = (int64_t)nsm;
    }
    c->stage2_applied = true;
    CUDA_TRY(c, tl.record(1, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    const float ms = tl.ms(0, 1);
    c->sstats.ms_final += ms;
    c->sstats.ms_total += ms;
    c->stage2_done = true;
    c->pos_valid = true;
    return ITSX_OK;
}
