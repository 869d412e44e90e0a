// cluster.cu -- greedy clustering of the exact derep classes at identity X < 1 on the GPU.
//
// Replaces `vsearch --cluster_size <seq> --id X --strand both --centroids rep.fa --uc uc.txt`
// (reference call site itsxpress/SeqSample.py:133-176).  Semantics (DESIGN.md §6):
//   classes are processed in a given order (abundance descending by default);
//   ed(a, b) is unit-cost Levenshtein distance over the derep's normalised residues, taken on both strands
//   (ed = min(ed(s_u, s_c), ed(rc(s_u), s_c)), '+' wins a tie);
//   with L = max(len_u, len_c) a pair is accepted iff (L - ed) / L >= X, i.e. iff ed <= D(L) (host table);
//   a class becomes a centroid iff no earlier centroid accepts it, else it joins the accepted earlier centroid of
//   highest identity (earliest on a tie).
//
// Kernels (all integer work on the resident reads; ranks r are positions in the processing order):
//   prep_kernel      per rank: first read, length, segment count; length histogram
//   seg_kernel       pigeonhole index: every class split into K(L)+1 segments, 64-bit key of (L, segment, residues)
//   query_kernel     per (rank, strand, partner length): every segment of that length looked up at shifts within
//                    +-D in the query strand; counts (pass 0) or emits (pass 1) candidates (u, v) with v earlier
//   verify_kernel    banded edit distance (band D) on both strands of every distinct candidate
//   round_kernel     greedy resolution over the accepted edges: one sweep per round until every class is decided
//   assign_kernel    each member's best centroid; remap kernels: centroid rows, read -> centroid row
//
// Losslessness: if ed(u, v) <= d with d <= K(len_v), at least one of the K(len_v)+1 segments of v is untouched by the
// alignment and occurs exactly in u's strand at its own position shifted by at most d.  Every such lookup is made, so
// no accepted pair is missed; a 64-bit key collision only adds a candidate that verification rejects.
//
// Per sample (sample ids set, per_sample = 1): a class is only ever compared with classes of its own sample.  The sample
// id seeds every segment key, so a template shared by many samples does not return one index hit per sample, and
// query_kernel drops any hit of another sample, so a key collision between samples never reaches verify_kernel (which
// would accept two similar sequences whatever their samples).  With no edge between samples, the rounds resolve every
// sample exactly as a call on that sample alone with the same relative order would.
#include <cub/cub.cuh>
#include "itsx_internal.h"

namespace {

constexpr int kMaxD = ITSX_CLUSTER_MAXD;

__device__ __forceinline__ uint32_t norm_c(uint32_t c)
{
    if (c >= 'a' && c <= 'z') c -= 32;
    return c == 'U' ? 'T' : c;
}
__device__ __forceinline__ uint32_t comp_c(uint32_t c)   // c normalised (derep.cu: comp_char)
{
    switch (c) {
        case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'T': return 'A';
        case 'R': return 'Y'; case 'Y': return 'R'; case 'M': return 'K'; case 'K': return 'M';
        case 'H': return 'D'; case 'D': return 'H'; case 'B': return 'V'; case 'V': return 'B';
        default: return c;
    }
}
// residue m of a read of length L on strand rc (0 '+', 1 '-')
__device__ __forceinline__ uint32_t res_at(const uint8_t *__restrict__ s, int L, int m, int rc)
{
    return rc ? comp_c(norm_c(s[L - 1 - m])) : norm_c(s[m]);
}
__device__ __forceinline__ unsigned long long mix64(unsigned long long k)
{
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull;
    k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull;
    k ^= k >> 33;
    return k;
}
// key of segment j of a class of length Lv in sample smp (0 without per-sample clustering: the keys of one sample are
// those of a call without samples): seg_key(seg_seed(Lv, j, smp), residues)
__device__ __forceinline__ unsigned long long seg_seed(int Lv, int j, int smp)
{
    return mix64(((unsigned long long)(uint32_t)smp << 40) ^ ((unsigned long long)Lv << 20) ^ (unsigned long long)j ^
                 0x9E3779B97F4A7C15ull);
}
__device__ __forceinline__ unsigned long long seg_key(unsigned long long h, const uint8_t *__restrict__ s, int L, int rc,
                                                      int q, int len)
{
    for (int m = 0; m < len; m++) h = (h ^ res_at(s, L, q + m, rc)) * 0x100000001b3ull;
    return mix64(h);
}
// segment j of k over a class of length L: [j*L/k, (j+1)*L/k); j*L/k = j*(L/k) + j*(L%k)/k exactly, in 32 bits (j <= k)
__device__ __forceinline__ int seg_lo(int L, int k, int j) { return j * (L / k) + j * (L % k) / k; }

inline unsigned nblk(int64_t n, int b) { return (unsigned)((n + b - 1) / b); }

// sample (per read) is null without per-sample clustering; rsample[r] is then 0
__global__ void prep_kernel(const int32_t *__restrict__ order, const int32_t *__restrict__ first,
                            const int64_t *__restrict__ off, const int32_t *__restrict__ K,
                            const int32_t *__restrict__ sample, int64_t nu, int32_t *__restrict__ rfirst,
                            int32_t *__restrict__ rlen, int32_t *__restrict__ rsample, int64_t *__restrict__ nseg,
                            int32_t *__restrict__ rank_of, int32_t *__restrict__ present)
{
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > nu) return;
    if (r == nu) { nseg[nu] = 0; return; }
    const int u = order[r], f = first[u];
    const int L = (int)(off[f + 1] - off[f]);
    rfirst[r] = f;
    rlen[r] = L;
    rsample[r] = sample ? sample[f] : 0;
    rank_of[u] = (int32_t)r;
    nseg[r] = L > 0 ? K[L] + 1 : 0;
    atomicAdd(&present[L], 1);
}

__global__ void seg_kernel(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ off,
                           const int32_t *__restrict__ rfirst, const int32_t *__restrict__ rlen,
                           const int32_t *__restrict__ rsample, const int64_t *__restrict__ segoff, int64_t nu,
                           unsigned long long kmask, unsigned long long *__restrict__ key, int32_t *__restrict__ val)
{
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nu) return;
    const int L = rlen[r];
    const int64_t o = segoff[r];
    const int k = (int)(segoff[r + 1] - o);
    const uint8_t *s = ascii + off[rfirst[r]];
    for (int j = 0; j < k; j++) {
        const int a = seg_lo(L, k, j), b = seg_lo(L, k, j + 1);
        key[o + j] = seg_key(seg_seed(L, j, rsample[r]), s, L, 0, a, b - a) & kmask;
        val[o + j] = (int32_t)r;
    }
}

// thread t = (rank, strand, partner-length slot); pass 0 counts the candidates of t, pass 1 writes them at out[base[t]].
// 10 blocks per SM leave ptxas room for the loop state without spills (left to itself it takes 32 registers and spills).
__global__ void __launch_bounds__(128, 10)
query_kernel(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ off, const int32_t *__restrict__ rfirst,
             const int32_t *__restrict__ rlen, const int32_t *__restrict__ rsample, int64_t nu, int W,
             const int32_t *__restrict__ D, const int32_t *__restrict__ K, const int32_t *__restrict__ lo,
             const int32_t *__restrict__ hi,
             const int32_t *__restrict__ present, const unsigned long long *__restrict__ skey,
             const int32_t *__restrict__ sval, int64_t nrec, unsigned long long kmask, int pass,
             int64_t *__restrict__ count,
             const int64_t *__restrict__ base, unsigned long long *__restrict__ out)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nu * 2 * W) return;
    const int t32 = (int)t;                                    // nu * 2 * W < 2^31 (cluster_run)
    const int r = t32 / (2 * W);
    const int rc = (t32 / W) & 1, slot = t32 % W;
    const int Lu = rlen[r];
    const int Lv = lo[Lu] + slot;
    int64_t n = 0;
    if (Lu > 0 && Lv > 0 && Lv <= hi[Lu] && present[Lv] > 0) {
        const uint8_t *s = ascii + off[rfirst[r]];
        const int d = D[max(Lu, Lv)], k = K[Lv] + 1, smp = rsample[r];
        int64_t w = pass ? base[t] : 0;
        for (int j = 0, a = 0, b; j < k; j++, a = b) {
            b = seg_lo(Lv, k, j + 1);
            const int len = b - a;
            const unsigned long long seed = seg_seed(Lv, j, smp);
            for (int q = max(0, a - d); q <= a + d && q + len <= Lu; q++) {
                const unsigned long long h = seg_key(seed, s, Lu, rc, q, len) & kmask;
                int64_t x = 0, y = nrec;                               // lower bound of h
                while (x < y) { const int64_t m = (x + y) >> 1; if (skey[m] < h) x = m + 1; else y = m; }
                for (; x < nrec && skey[x] == h; x++) {
                    const int32_t v = sval[x];
                    if (v >= r || rsample[v] != smp) continue;
                    if (pass) out[w++] = ((unsigned long long)r << 32) | (uint32_t)v;
                    n++;
                }
            }
        }
    }
    if (!pass) count[t] = n;
}

// banded unit-cost edit distance of t (length n, strand rc of read s) against v (length m, '+'); d+1 if above d
__device__ int banded_ed(const uint8_t *__restrict__ s, int n, int rc, const uint8_t *__restrict__ v, int m, int d)
{
    if (abs(n - m) > d) return d + 1;
    const int INF = d + 1;
    uint8_t row[2 * kMaxD + 2];          // row[k] = cell (i, j = i + k - d), capped at d + 1
    for (int k = 0; k <= 2 * d + 1; k++) row[k] = (uint8_t)((k >= d && k - d <= m && k <= 2 * d) ? k - d : INF);
    for (int i = 1; i <= n; i++) {
        const uint32_t ti = res_at(s, n, i - 1, rc);
        int left = INF, best = INF;
        for (int k = 0; k <= 2 * d; k++) {
            const int j = i + k - d;
            int x = INF;
            if (j >= 0 && j <= m) {
                x = row[k + 1] + 1;                                          // (i-1, j)
                if (j > 0) {
                    x = min(x, row[k] + (ti != norm_c(v[j - 1]) ? 1 : 0));   // (i-1, j-1)
                    x = min(x, left + 1);                                    // (i, j-1)
                }
                x = min(x, INF);
            }
            row[k] = (uint8_t)x;
            left = x;
            best = min(best, x);
        }
        if (best > d) return INF;
    }
    return row[m - n + d];
}

// acc[e] = the pair is accepted; edinfo[e] = ed | 0x80 when the '-' strand is strictly closer
__global__ void __launch_bounds__(128)
verify_kernel(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ off, const int32_t *__restrict__ rfirst,
              const int32_t *__restrict__ rlen, const int32_t *__restrict__ D, const unsigned long long *__restrict__ cand,
              int64_t ncand, uint8_t *__restrict__ acc, uint8_t *__restrict__ edinfo)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= ncand) return;
    const int u = (int)(cand[e] >> 32), v = (int)(cand[e] & 0xffffffffu);
    const int Lu = rlen[u], Lv = rlen[v], d = D[max(Lu, Lv)];
    const uint8_t *su = ascii + off[rfirst[u]], *sv = ascii + off[rfirst[v]];
    const int ep = banded_ed(su, Lu, 0, sv, Lv, d);
    const int em = ep == 0 ? ep : banded_ed(su, Lu, 1, sv, Lv, min(d, ep));
    const int ed = min(ep, em);
    acc[e] = ed <= d;
    edinfo[e] = (uint8_t)(ed | (em < ep ? 0x80 : 0));
}

__global__ void edge_begin_kernel(const unsigned long long *__restrict__ edge, int64_t ne, int64_t nu,
                                  int64_t *__restrict__ beg)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > nu) return;
    int64_t x = 0, y = ne;
    while (x < y) { const int64_t m = (x + y) >> 1; if ((int64_t)(edge[m] >> 32) < r) x = m + 1; else y = m; }
    beg[r] = x;
}

enum { UNDECIDED = 0, CENTROID = 1, MEMBER = 2 };

__global__ void round_kernel(const unsigned long long *__restrict__ edge, const int64_t *__restrict__ beg, int64_t nu,
                             volatile uint8_t *state, unsigned long long *__restrict__ undecided)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nu || state[r] != UNDECIDED) return;
    bool all_members = true;
    for (int64_t x = beg[r]; x < beg[r + 1]; x++) {
        const uint8_t sv = state[edge[x] & 0xffffffffu];
        if (sv == CENTROID) { state[r] = MEMBER; return; }
        if (sv != MEMBER) all_members = false;
    }
    if (all_members) state[r] = CENTROID;
    else atomicAdd(undecided, 1ull);
}

// best centroid of every rank (itself for a centroid): highest (L - ed) / L by cross-multiplication, earliest on a tie
__global__ void assign_kernel(const unsigned long long *__restrict__ edge, const uint8_t *__restrict__ edinfo,
                              const int64_t *__restrict__ beg, const int32_t *__restrict__ rlen, const uint8_t *__restrict__ state,
                              int64_t nu, int32_t *__restrict__ cent, uint8_t *__restrict__ strand, int32_t *__restrict__ edout)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nu) return;
    int32_t best = (int32_t)r, bed = 0;
    uint8_t bst = 0;
    if (state[r] == MEMBER) {
        best = -1;
        long long bn = 0, bd = 1;
        for (int64_t x = beg[r]; x < beg[r + 1]; x++) {
            const int v = (int)(edge[x] & 0xffffffffu);
            if (state[v] != CENTROID) continue;
            const int ed = edinfo[x] & 0x7f;
            const long long L = max(rlen[r], rlen[v]), num = L - ed;
            if (best < 0 || num * bd > bn * L) { best = v; bn = num; bd = L; bed = ed; bst = edinfo[x] >> 7; }
        }
    }
    cent[r] = best;
    strand[r] = bst;
    edout[r] = bed;
}

__global__ void is_centroid_kernel(const uint8_t *__restrict__ state, int64_t nu, int32_t *__restrict__ flag)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < nu) flag[r] = state[r] == CENTROID;
}
// per class u: centroid row, strand and ed; per centroid row: its class and its first read (the search set)
__global__ void remap_unique_kernel(const int32_t *__restrict__ order, const int32_t *__restrict__ rcent,
                                    const uint8_t *__restrict__ rstrand, const int32_t *__restrict__ red,
                                    const int32_t *__restrict__ row_of_rank, const uint8_t *__restrict__ state,
                                    const int32_t *__restrict__ first, int64_t nu, int32_t *__restrict__ crow,
                                    uint8_t *__restrict__ cstrand, int32_t *__restrict__ ced,
                                    int32_t *__restrict__ unique_of_row, int32_t *__restrict__ first_of_row)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nu) return;
    const int u = order[r];
    crow[u] = row_of_rank[rcent[r]];
    cstrand[u] = rstrand[r];
    ced[u] = red[r];
    if (state[r] == CENTROID) {
        unique_of_row[row_of_rank[r]] = u;
        first_of_row[row_of_rank[r]] = first[u];
    }
}
__global__ void remap_read_kernel(const int32_t *__restrict__ class_uid, const int32_t *__restrict__ crow, int64_t n,
                                  int32_t *__restrict__ uid)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) uid[i] = crow[class_uid[i]];
}

// per unique: length and abundance (the derep counts a class at its first read); iota for the default order
__global__ void unique_kernel(const int32_t *__restrict__ first, const int64_t *__restrict__ off,
                              const int32_t *__restrict__ abund, int64_t nu, int32_t *__restrict__ len,
                              int32_t *__restrict__ ab, int32_t *__restrict__ iota)
{
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= nu) return;
    const int f = first[u];
    len[u] = (int32_t)(off[f + 1] - off[f]);
    ab[u] = abund[f];
    iota[u] = (int32_t)u;
}

}  // namespace


void cluster_dtable(double id, int32_t lmax, int32_t *D)
{
    for (int32_t L = 0; L <= lmax; L++) {
        int32_t e = 0;
        while (e < L && (double)(L - (e + 1)) / (double)L >= id) e++;
        D[L] = e;
    }
}

int cluster_run(itsx_ctx *c, const itsx_cluster_params *prm, const int32_t *order_in, int64_t *n_centroids)
{
    cudaStream_t st = c->stream;
    const int64_t nu = c->n_unique, n = c->nreads;
    if (!prm || !(prm->id > 0.5 && prm->id <= 1.0)) { c->err = "cluster: id must be in (0.5, 1]"; return ITSX_EINVAL; }
    if (!prm->strand_both) { c->err = "cluster: only strand_both = 1 (the derep classes are strand-independent)"; return ITSX_EINVAL; }
    if (c->map_external || c->stream_open || c->dstats.n_reads != c->nreads || c->dstats.n_unique != nu) {
        c->err = "cluster: no dereplicated reads are resident (itsx_derep / itsx_derep_resident first)";
        return ITSX_EINVAL;
    }
    if (c->have_samples && !prm->per_sample) {
        c->err = "cluster: the reads carry sample ids (set per_sample to cluster each sample on its own)";
        return ITSX_EINVAL;
    }
    if (nu >= (1ll << 31) - 1) { c->err = "cluster: more than 2^31-2 unique sequences"; return ITSX_ELIMIT; }
    itsx_cluster_stats cs{};
    cs.n_unique = nu;
    // the exact class of every read survives re-clustering the same derep (d_uid is rewritten at the end)
    if (!c->cl_active) {
        CUDA_TRY(c, c->d_cl_class.ensure((size_t)std::max<int64_t>(n, 1) * 4));
        if (n) CUDA_TRY(c, cudaMemcpyAsync(c->d_cl_class.p, c->d_uid.p, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
    }
    Timeline<6> tl;     // ends of set-up + index, candidates, dedup + verify, resolution, remap
    CUDA_TRY(c, tl.status);
    CUDA_TRY(c, tl.record(0, st));
    const size_t nu1 = (size_t)std::max<int64_t>(nu, 1);
    const int32_t *first = c->d_first.as<int32_t>();
    const int64_t *off = c->d_off.as<int64_t>();
    const uint8_t *ascii = c->d_ascii.as<uint8_t>();

    // ---- set-up: lengths, abundance, processing order, the D / K / lo / hi tables -----------------------------------
    CUDA_TRY(c, c->d_cl_order.ensure(nu1 * 4));
    CUDA_TRY(c, c->d_cl_u.ensure(nu1 * 4 * 4));
    int32_t *order = c->d_cl_order.as<int32_t>();
    int32_t *ulen = c->d_cl_u.as<int32_t>(), *uab = ulen + nu1, *uab2 = uab + nu1, *iota = uab2 + nu1;
    CUDA_TRY(c, c->d_counters.ensure(64 * 8));
    int32_t *d_max = (int32_t *)(c->d_counters.as<unsigned long long>() + 48);
    unsigned long long *d_undec = c->d_counters.as<unsigned long long>() + 49;
    int32_t lmax = 0;
    if (nu) {
        unique_kernel<<<nblk(nu, 256), 256, 0, st>>>(first, off, c->d_abund.as<int32_t>(), nu, ulen, uab, iota);
        c->launches++;
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceReduce::Max(t, b, ulen, d_max, (int)nu, st); }));
        CUDA_TRY(c, cudaMemcpyAsync(&lmax, d_max, 4, cudaMemcpyDeviceToHost, st));
        if (order_in) {
            std::vector<int32_t> h((size_t)nu);
            CUDA_TRY(c, cudaMemcpyAsync(h.data(), order_in, (size_t)nu * 4, cudaMemcpyDefault, st));
            CUDA_TRY(c, cudaStreamSynchronize(st));
            std::vector<char> seen((size_t)nu, 0);
            for (int32_t u : h) {
                if (u < 0 || u >= nu || seen[u]) { c->err = "cluster: order is not a permutation of the unique indices"; return ITSX_EINVAL; }
                seen[u] = 1;
            }
            CUDA_TRY(c, cudaMemcpyAsync(order, h.data(), (size_t)nu * 4, cudaMemcpyHostToDevice, st));
        } else {
            // abundance descending, then first occurrence (= unique index) ascending: the radix sort is stable
            CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) {
                return cub::DeviceRadixSort::SortPairsDescending(t, b, uab, uab2, iota, order, (int)nu, 0, 32, st);
            }));
        }
        CUDA_TRY(c, cudaStreamSynchronize(st));
    }
    std::vector<int32_t> tab(4 * ((size_t)lmax + 1));
    int32_t *D = tab.data(), *K = D + lmax + 1, *LO = K + lmax + 1, *HI = LO + lmax + 1;
    cluster_dtable(prm->id, lmax, D);
    cs.d_max = D[lmax];
    if (D[lmax] > ITSX_CLUSTER_MAXD) {
        c->err = "cluster: the longest unique sequence allows more than ITSX_CLUSTER_MAXD edits at this identity";
        return ITSX_ELIMIT;
    }
    int W = 1;
    for (int32_t L = 0, hi = 0; L <= lmax; L++) {
        while (hi + 1 <= lmax && (hi + 1) - D[hi + 1] <= L) hi++;   // L - D(L) is non-decreasing
        HI[L] = std::max(hi, L);
        LO[L] = L - D[L];
        K[L] = D[HI[L]];          // the largest band of any pair with a class of length L (D is non-decreasing)
        W = std::max(W, HI[L] - LO[L] + 1);
    }
    cs.n_len_slots = W;
    CUDA_TRY(c, c->d_cl_tab.ensure(tab.size() * 4 + ((size_t)lmax + 1) * 4));
    int32_t *dD = c->d_cl_tab.as<int32_t>(), *dK = dD + lmax + 1, *dLO = dK + lmax + 1, *dHI = dLO + lmax + 1;
    int32_t *present = dHI + lmax + 1;
    CUDA_TRY(c, cudaMemcpyAsync(dD, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemsetAsync(present, 0, ((size_t)lmax + 1) * 4, st));

    // ---- pigeonhole index: K(L)+1 segments per class, sorted by key ------------------------------------------------
    CUDA_TRY(c, c->d_cl_r.ensure(nu1 * 4 * 4));
    int32_t *rfirst = c->d_cl_r.as<int32_t>(), *rlen = rfirst + nu1, *rank_of = rlen + nu1, *rsample = rank_of + nu1;
    const int32_t *sample = c->have_samples ? c->d_sample.as<int32_t>() : nullptr;
    CUDA_TRY(c, c->d_cl_seg.ensure((nu1 + 1) * 8 * 2));
    int64_t *nseg = c->d_cl_seg.as<int64_t>(), *segoff = nseg + nu1 + 1;
    int64_t nrec = 0;
    const unsigned long long kmask = c->cl_key_bits >= 64 ? ~0ull : ((1ull << c->cl_key_bits) - 1ull);
    if (nu) {
        prep_kernel<<<nblk(nu + 1, 256), 256, 0, st>>>(order, first, off, dK, sample, nu, rfirst, rlen, rsample, nseg,
                                                       rank_of, present);
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, nseg, segoff, (int)nu + 1, st); }));
        CUDA_TRY(c, cudaMemcpyAsync(&nrec, segoff + nu, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        c->launches++;
    }
    if (nrec >= (1ll << 31)) { c->err = "cluster: more than 2^31-1 index segments"; return ITSX_ELIMIT; }
    CUDA_TRY(c, c->d_cl_key.ensure((size_t)std::max<int64_t>(nrec, 1) * 8 * 2));
    CUDA_TRY(c, c->d_cl_val.ensure((size_t)std::max<int64_t>(nrec, 1) * 4 * 2));
    unsigned long long *key = c->d_cl_key.as<unsigned long long>(), *skey = key + std::max<int64_t>(nrec, 1);
    int32_t *val = c->d_cl_val.as<int32_t>(), *sval = val + std::max<int64_t>(nrec, 1);
    if (nrec) {
        seg_kernel<<<nblk(nu, 128), 128, 0, st>>>(ascii, off, rfirst, rlen, rsample, segoff, nu, kmask, key, val);
        c->launches++;
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) {
            return cub::DeviceRadixSort::SortPairs(t, b, key, skey, val, sval, (int)nrec, 0, 64, st);
        }));
    }
    cs.n_segments = nrec;
    CUDA_TRY(c, tl.record(1, st));

    // ---- candidates: count, scan, emit ------------------------------------------------------------------------------
    const int64_t T = nu * 2 * (int64_t)W;
    if (T + 1 >= (1ll << 31)) { c->err = "cluster: too many (sequence, strand, length) lookups in one call"; return ITSX_ELIMIT; }
    CUDA_TRY(c, c->d_cl_cnt.ensure((size_t)(T + 1) * 8 * 2));
    int64_t *cnt = c->d_cl_cnt.as<int64_t>(), *cbase = cnt + T + 1;
    int64_t ncand = 0;
    if (nrec) {
        query_kernel<<<nblk(T, 128), 128, 0, st>>>(ascii, off, rfirst, rlen, rsample, nu, W, dD, dK, dLO, dHI, present,
                                                   skey, sval, nrec, kmask, 0, cnt, nullptr, nullptr);
        CUDA_TRY(c, cudaMemsetAsync(cnt + T, 0, 8, st));
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, cnt, cbase, (int)T + 1, st); }));
        CUDA_TRY(c, cudaMemcpyAsync(&ncand, cbase + T, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        c->launches++;
    }
    if (ncand >= (1ll << 31)) { c->err = "cluster: more than 2^31-1 candidate pairs"; return ITSX_ELIMIT; }
    const size_t nc1 = (size_t)std::max<int64_t>(ncand, 1);
    CUDA_TRY(c, c->d_cl_cand.ensure(nc1 * 8 * 2));
    unsigned long long *cand = c->d_cl_cand.as<unsigned long long>(), *cand2 = cand + nc1;
    if (ncand) {
        query_kernel<<<nblk(T, 128), 128, 0, st>>>(ascii, off, rfirst, rlen, rsample, nu, W, dD, dK, dLO, dHI, present,
                                                   skey, sval, nrec, kmask, 1, nullptr, cbase, cand);
        c->launches++;
    }
    cs.n_candidates = ncand;
    CUDA_TRY(c, tl.record(2, st));

    // ---- distinct pairs (sorted by (u, v)), verification, accepted edges --------------------------------------------
    CUDA_TRY(c, c->d_cl_acc.ensure(nc1 * 2));
    uint8_t *acc = c->d_cl_acc.as<uint8_t>(), *edinfo = acc + nc1;
    CUDA_TRY(c, c->d_cl_edge.ensure(nc1 * 9));
    unsigned long long *edge = c->d_cl_edge.as<unsigned long long>();
    uint8_t *einfo = (uint8_t *)(edge + nc1);
    int64_t *d_nsel = (int64_t *)(c->d_counters.as<unsigned long long>() + 50);
    int64_t nver = 0, nacc = 0;
    if (ncand) {
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceRadixSort::SortKeys(t, b, cand, cand2, (int)ncand, 0, 64, st); }));
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceSelect::Unique(t, b, cand2, cand, d_nsel, (int)ncand, st); }));
        CUDA_TRY(c, cudaMemcpyAsync(&nver, d_nsel, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        verify_kernel<<<nblk(nver, 128), 128, 0, st>>>(ascii, off, rfirst, rlen, dD, cand, nver, acc, edinfo);
        c->launches++;
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceSelect::Flagged(t, b, cand, acc, edge, d_nsel, (int)nver, st); }));
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceSelect::Flagged(t, b, edinfo, acc, einfo, d_nsel, (int)nver, st); }));
        CUDA_TRY(c, cudaMemcpyAsync(&nacc, d_nsel, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
    }
    cs.n_verified = nver;
    cs.n_accepted = nacc;
    CUDA_TRY(c, tl.record(3, st));

    // ---- greedy resolution in rounds, then every member's best centroid ----------------------------------------------
    CUDA_TRY(c, c->d_cl_beg.ensure((nu1 + 1) * 8));
    int64_t *beg = c->d_cl_beg.as<int64_t>();
    CUDA_TRY(c, c->d_cl_state.ensure(nu1));
    uint8_t *state = c->d_cl_state.as<uint8_t>();
    CUDA_TRY(c, c->d_cl_rres.ensure(nu1 * 9));
    int32_t *rcent = c->d_cl_rres.as<int32_t>(), *red = rcent + nu1;
    uint8_t *rstrand = (uint8_t *)(red + nu1);
    if (nu) {
        edge_begin_kernel<<<nblk(nu + 1, 256), 256, 0, st>>>(edge, nacc, nu, beg);
        CUDA_TRY(c, cudaMemsetAsync(state, UNDECIDED, (size_t)nu, st));
        c->launches++;
        for (unsigned long long undecided = 1; undecided;) {
            if (cs.n_rounds > nu) { c->err = "cluster: the resolution made no progress"; return ITSX_ELIMIT; }
            CUDA_TRY(c, cudaMemsetAsync(d_undec, 0, 8, st));
            round_kernel<<<nblk(nu, 256), 256, 0, st>>>(edge, beg, nu, state, d_undec);
            CUDA_TRY(c, cudaMemcpyAsync(&undecided, d_undec, 8, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(c, cudaStreamSynchronize(st));
            c->launches++;
            cs.n_rounds++;
        }
        assign_kernel<<<nblk(nu, 256), 256, 0, st>>>(edge, einfo, beg, rlen, state, nu, rcent, rstrand, red);
        c->launches++;
    }
    CUDA_TRY(c, tl.record(4, st));

    // ---- remap: centroid rows in processing order, per-unique results, read -> centroid row, the search set ----------
    CUDA_TRY(c, c->d_cl_row.ensure((nu1 + 1) * 4 * 2));
    int32_t *cflag = c->d_cl_row.as<int32_t>(), *row_of_rank = cflag + nu1 + 1;
    CUDA_TRY(c, c->d_cl_out.ensure(nu1 * 9));
    int32_t *crow = c->d_cl_out.as<int32_t>(), *ced = crow + nu1;
    uint8_t *cstrand = (uint8_t *)(ced + nu1);
    int32_t ncent = 0;
    if (nu) {
        is_centroid_kernel<<<nblk(nu, 256), 256, 0, st>>>(state, nu, cflag);
        CUDA_TRY(c, cudaMemsetAsync(cflag + nu, 0, 4, st));
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, cflag, row_of_rank, (int)nu + 1, st); }));
        CUDA_TRY(c, cudaMemcpyAsync(&ncent, row_of_rank + nu, 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
    }
    CUDA_TRY(c, c->d_cl_crow.ensure((size_t)std::max(ncent, 1) * 4 * 2));
    int32_t *unique_of_row = c->d_cl_crow.as<int32_t>(), *first_of_row = unique_of_row + std::max(ncent, 1);
    if (nu) {
        remap_unique_kernel<<<nblk(nu, 256), 256, 0, st>>>(order, rcent, rstrand, red, row_of_rank, state, first, nu, crow,
                                                           cstrand, ced, unique_of_row, first_of_row);
        remap_read_kernel<<<nblk(n, 256), 256, 0, st>>>(c->d_cl_class.as<int32_t>(), crow, n, c->d_uid.as<int32_t>());
        c->launches += 3;
    }
    int rc = search_build_seqs_from_reads(c, first_of_row, ncent);
    if (rc) return rc;
    CUDA_TRY(c, tl.record(5, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    cs.n_centroids = ncent;
    cs.ms_index = tl.ms(0, 1);
    cs.ms_candidates = tl.ms(1, 2);
    cs.ms_verify = tl.ms(2, 3);
    cs.ms_resolve = tl.ms(3, 4);
    cs.ms_remap = tl.ms(4, 5);
    cs.ms_total = tl.ms(0, 5);
    c->clstats = cs;
    c->cl_active = true;
    c->cl_ncent = ncent;
    if (n_centroids) *n_centroids = ncent;
    return ITSX_OK;
}
