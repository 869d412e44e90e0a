// derep.cu -- exact full-length dereplication over both strands on the GPU.
//
// Replaces `vsearch --fastx_uniques <fq> --fastaout rep.fa --uc uc.txt --strand both`
// (reference call site itsxpress/SeqSample.py:93-131) and the read -> representative map that
// Dedup.parse rebuilds from uc.txt (SeqSample.py:542-562).  Semantics (SURVEY.md Appendix B):
// case-insensitive, U == T, IUPAC letters are ordinary symbols, a read joins the class of an
// earlier read that equals it or its reverse complement, the representative is the FIRST read
// of the class in input order.
//
// Kernels (all HBM/L2-bound integer work, no tensor cores):
//   pack2_kernel      ASCII -> 2-bit stream (16 bases / u32) + non-ACGT bit mask; 16 B per thread,
//                     perfectly coalesced, independent of read boundaries.
//   hash_kernel       per read: canonical orientation (word-wise compare of s and revcomp(s)),
//                     murmur-style 64-bit key over the canonical 2-bit words (+ length).
//   insert_kernel     open-addressing table in HBM: atomicCAS on the key, atomicMin on the first index.
//   verify_kernel     full-sequence compare of every read with its slot's first read; abundance
//                     counts; mismatches (64-bit collisions) go to a list ...
//   collide_kernel    ... that is resolved exactly among themselves (all-pairs; normally empty).
//   uniq kernels      representatives -> dense unique ids in first-occurrence order.
#include <cub/cub.cuh>
#include "itsx_internal.h"

namespace {

constexpr unsigned long long kEmpty = ~0ull;
struct Slot {
    unsigned long long key;
    int first;
    int pad;
};

#define FLAG_EXC 1u
#define FLAG_RC 2u

// ---- K1a: ASCII -> 2-bit + exception mask --------------------------------------------------
__device__ __forceinline__ uint32_t pack4(uint32_t w, uint32_t &bad)
{
    uint32_t t = ((w >> 1) ^ (w >> 2)) & 0x03030303u;            // A,C,G,T/U -> 0,1,2,3 (any case)
    uint32_t u = w & 0xDFDFDFDFu;                                  // fold case
    uint32_t ok = __vcmpeq4(u, 0x41414141u) | __vcmpeq4(u, 0x43434343u) | __vcmpeq4(u, 0x47474747u) |
                  __vcmpeq4(u, 0x54545454u) | __vcmpeq4(u, 0x55555555u);
    uint32_t b = (~ok) & 0x01010101u;
    bad = (b | (b >> 7) | (b >> 14) | (b >> 21)) & 0xFu;
    t &= ok & 0x03030303u;                                         // exceptions pack as 0
    return (t | (t >> 6) | (t >> 12) | (t >> 18)) & 0xFFu;
}

__global__ void __launch_bounds__(256) pack2_kernel(const uint4 *__restrict__ ascii, int64_t nchunk,
                                                    uint32_t *__restrict__ pack2, uint16_t *__restrict__ exc)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nchunk) return;
    uint4 v = __ldg(ascii + i);
    uint32_t b0, b1, b2, b3;
    uint32_t p = pack4(v.x, b0) | (pack4(v.y, b1) << 8) | (pack4(v.z, b2) << 16) | (pack4(v.w, b3) << 24);
    pack2[i] = p;
    exc[i]   = (uint16_t)(b0 | (b1 << 4) | (b2 << 8) | (b3 << 12));
}

// ---- 2-bit word access -----------------------------------------------------------------------
__device__ __forceinline__ uint32_t extract16(const uint32_t *__restrict__ P, int64_t pos)
{
    int64_t idx = pos >> 4;
    int sh = (int)(pos & 15) * 2;
    return __funnelshift_r(P[idx], P[idx + 1], sh);
}
__device__ __forceinline__ uint32_t pairrev(uint32_t x)
{
    x = __brev(x);
    return ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
}
__device__ __forceinline__ uint32_t fwd_word(const uint32_t *__restrict__ P, int64_t base, int j, int L)
{
    uint32_t w = extract16(P, base + 16 * j);
    int rem = L - 16 * j;
    if (rem < 16) w &= (1u << (2 * rem)) - 1u;
    return w;
}
__device__ __forceinline__ uint32_t rc_word(const uint32_t *__restrict__ P, int64_t base, int j, int L)
{
    int end = L - 16 * j, start = end - 16;
    if (start >= 0) return ~pairrev(extract16(P, base + start));
    uint32_t u = extract16(P, base) << (2 * (16 - end));
    return (~pairrev(u)) & ((1u << (2 * end)) - 1u);
}
__device__ __forceinline__ uint32_t canon_word(const uint32_t *__restrict__ P, int64_t base, int j, int L, bool rc)
{
    return rc ? rc_word(P, base, j, L) : fwd_word(P, base, j, L);
}

// ---- byte path for reads that contain non-ACGT symbols ----------------------------------------
__device__ __forceinline__ uint32_t norm_char(uint32_t c)
{
    if (c >= 'a' && c <= 'z') c -= 32;
    return c == 'U' ? 'T' : c;
}
__device__ uint32_t comp_char(uint32_t c)   // c normalised
{
    switch (c) {
        case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'T': return 'A';
        case 'R': return 'Y'; case 'Y': return 'R'; case 'M': return 'K'; case 'K': return 'M';
        case 'H': return 'D'; case 'D': return 'H'; case 'B': return 'V'; case 'V': return 'B';
        default: return c;   // S, W, N and anything else map to themselves
    }
}
__device__ __forceinline__ uint32_t canon_char(const uint8_t *__restrict__ s, int m, int L, bool rc)
{
    return rc ? comp_char(norm_char(s[L - 1 - m])) : norm_char(s[m]);
}

__device__ __forceinline__ unsigned long long mix64(unsigned long long k)
{
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull;
    k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull;
    k ^= k >> 33;
    return k;
}
__device__ __forceinline__ unsigned long long rotl64(unsigned long long x, int r) { return (x << r) | (x >> (64 - r)); }

__device__ bool range_has_exc(const uint16_t *__restrict__ exc, int64_t base, int L)
{
    int64_t c0 = base >> 4, c1 = (base + L - 1) >> 4;
    for (int64_t c = c0; c <= c1; c++) {
        uint32_t m = exc[c];
        if (c == c0) m &= 0xFFFFu << (base & 15);
        if (c == c1) m &= 0xFFFFu >> (15 - ((base + L - 1) & 15));
        if (m & 0xFFFFu) return true;
    }
    return false;
}

// ---- K1b: canonical orientation + 64-bit key ---------------------------------------------------
__global__ void __launch_bounds__(128) hash_kernel(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ off,
                                                   const uint32_t *__restrict__ P, const uint16_t *__restrict__ exc,
                                                   int64_t nreads, unsigned long long keymask,
                                                   const int32_t *__restrict__ sample,
                                                   unsigned long long *__restrict__ key, uint8_t *__restrict__ flags)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nreads) return;
    const int64_t base = off[i];
    const int L = (int)(off[i + 1] - base);
    unsigned long long h = 0x9E3779B97F4A7C15ull ^ ((unsigned long long)L * 0x87c37b91114253d5ull);
    uint32_t fl = 0;
    if (L > 0 && range_has_exc(exc, base, L)) {
        fl = FLAG_EXC;
        const uint8_t *s = ascii + base;
        bool rc = false;
        for (int m = 0; m < L; m++) {
            uint32_t a = norm_char(s[m]), b = comp_char(norm_char(s[L - 1 - m]));
            if (a != b) { rc = b < a; break; }
        }
        if (rc) fl |= FLAG_RC;
        h ^= 0x5bd1e9955bd1e995ull;
        for (int m = 0; m < L; m++) {
            h ^= canon_char(s, m, L, rc);
            h *= 0x100000001b3ull;
            h = rotl64(h, 23);
        }
    } else if (L > 0) {
        const int nw = (L + 15) >> 4;
        bool rc = false;
        for (int j = 0; j < nw; j++) {
            uint32_t f = fwd_word(P, base, j, L), r = rc_word(P, base, j, L);
            if (f != r) { rc = r < f; break; }
        }
        if (rc) fl |= FLAG_RC;
        int j = 0;
        for (; j + 1 < nw; j += 2) {
            unsigned long long k = (unsigned long long)canon_word(P, base, j, L, rc) |
                                   ((unsigned long long)canon_word(P, base, j + 1, L, rc) << 32);
            k *= 0x87c37b91114253d5ull; k = rotl64(k, 31); k *= 0x4cf5ad432745937full;
            h ^= k; h = rotl64(h, 27) * 5ull + 0x52dce729ull;
        }
        if (j < nw) {
            unsigned long long k = canon_word(P, base, j, L, rc);
            k *= 0x87c37b91114253d5ull; k = rotl64(k, 31); k *= 0x4cf5ad432745937full;
            h ^= k; h = rotl64(h, 27) * 5ull + 0x52dce729ull;
        }
    }
    if (sample) h ^= mix64((unsigned long long)(uint32_t)sample[i] * 0x9E3779B97F4A7C15ull + 0x632BE59BD9B4E019ull);
    h = mix64(h) & keymask;
    if (h == kEmpty) h = 0x7fffffffffffffffull;
    key[i]   = h;
    flags[i] = (uint8_t)fl;
}

// ---- K2a: insert ------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) insert_kernel(const unsigned long long *__restrict__ key, int64_t nreads,
                                                     Slot *__restrict__ table, unsigned long long mask)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nreads) return;
    const unsigned long long k = key[i];
    unsigned long long s = mix64(k ^ 0xD6E8FEB86659FD93ull) & mask;
    while (true) {
        unsigned long long prev = atomicCAS(&table[s].key, kEmpty, k);
        if (prev == kEmpty || prev == k) {
            atomicMin(&table[s].first, (int)i);
            return;
        }
        s = (s + 1) & mask;
    }
}

__device__ bool same_class(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ off,
                           const uint32_t *__restrict__ P, const uint8_t *__restrict__ flags,
                           const int32_t *__restrict__ sample, int64_t a, int64_t b)
{
    if (sample && sample[a] != sample[b]) return false;      // classes never span samples
    const int64_t ba = off[a], bb = off[b];
    const int L = (int)(off[a + 1] - ba);
    if ((int)(off[b + 1] - bb) != L) return false;
    const uint32_t fa = flags[a], fb = flags[b];
    if ((fa ^ fb) & FLAG_EXC) return false;
    const bool ra = fa & FLAG_RC, rb = fb & FLAG_RC;
    if (fa & FLAG_EXC) {
        for (int m = 0; m < L; m++)
            if (canon_char(ascii + ba, m, L, ra) != canon_char(ascii + bb, m, L, rb)) return false;
        return true;
    }
    const int nw = (L + 15) >> 4;
    for (int j = 0; j < nw; j++)
        if (canon_word(P, ba, j, L, ra) != canon_word(P, bb, j, L, rb)) return false;
    return true;
}

// ---- K2b: verify against the slot's first read, count abundance -----------------------------------
__global__ void __launch_bounds__(128) verify_kernel(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ off,
                                                     const uint32_t *__restrict__ P,
                                                     const unsigned long long *__restrict__ key,
                                                     const uint8_t *__restrict__ flags, const int32_t *__restrict__ sample,
                                                     int64_t nreads,
                                                     const Slot *__restrict__ table, unsigned long long mask,
                                                     int32_t *__restrict__ rep, uint8_t *__restrict__ strand,
                                                     int32_t *__restrict__ abund, int32_t *__restrict__ collide,
                                                     unsigned long long *__restrict__ ncollide)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nreads) return;
    const unsigned long long k = key[i];
    unsigned long long s = mix64(k ^ 0xD6E8FEB86659FD93ull) & mask;
    while (table[s].key != k) s = (s + 1) & mask;
    const int r = table[s].first;
    if (r == (int)i || same_class(ascii, off, P, flags, sample, i, r)) {
        rep[i]    = r;
        strand[i] = ((flags[i] ^ flags[r]) & FLAG_RC) ? 1 : 0;
        atomicAdd(&abund[r], 1);
    } else {
        unsigned long long slot = atomicAdd(ncollide, 1ull);
        collide[slot] = (int32_t)i;
        rep[i] = -1;
    }
}

// ---- rare path: exact all-pairs resolution among collided reads -------------------------------------
__global__ void collide_kernel(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ off,
                               const uint32_t *__restrict__ P, const uint8_t *__restrict__ flags,
                               const int32_t *__restrict__ sample,
                               const int32_t *__restrict__ collide, int64_t nc, int32_t *__restrict__ rep,
                               uint8_t *__restrict__ strand, int32_t *__restrict__ abund)
{
    int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nc) return;
    const int a = collide[t];
    int best = a;
    for (int64_t u = 0; u < nc; u++) {
        const int b = collide[u];
        if (b < best && same_class(ascii, off, P, flags, sample, a, b)) best = b;
    }
    rep[a]    = best;
    strand[a] = ((flags[a] ^ flags[best]) & FLAG_RC) ? 1 : 0;
    atomicAdd(&abund[best], 1);
}

// ---- K3: dense unique ids in first-occurrence order ---------------------------------------------------
__global__ void isrep_kernel(const int32_t *__restrict__ rep, int64_t n, int32_t *__restrict__ flag)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = rep[i] == (int32_t)i;
}
__global__ void first_kernel(const int32_t *__restrict__ rep, const int32_t *__restrict__ scan, int64_t n,
                             int32_t *__restrict__ first)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && rep[i] == (int32_t)i) first[scan[i]] = (int32_t)i;
}
__global__ void uid_kernel(const int32_t *__restrict__ rep, const int32_t *__restrict__ scan, int64_t n,
                           int32_t *__restrict__ uid)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) uid[i] = scan[rep[i]];
}
__global__ void table_init_kernel(Slot *t, int64_t n)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { t[i].key = kEmpty; t[i].first = 0x7fffffff; t[i].pad = 0; }
}

inline unsigned nblk(int64_t n, int b) { return (unsigned)((n + b - 1) / b); }

}  // namespace

int derep_run(itsx_ctx *c)
{
    cudaStream_t st = c->stream;
    const int64_t n = c->nreads, total = c->total_bases;
    itsx_derep_stats &ds = c->dstats;
    ds = itsx_derep_stats{};
    ds.n_reads = n;
    ds.bytes_ascii = total;
    c->n_unique = 0;
    c->cl_active = false;
    if (n == 0) return ITSX_OK;
    if (n >= 0x7fffffffLL) { c->err = "derep: more than 2^31-1 reads in one call"; return ITSX_ELIMIT; }

    const int64_t nchunk = (total + 15) / 16;
    CUDA_TRY(c, c->d_pack2.ensure((size_t)(nchunk + 2) * 4));
    CUDA_TRY(c, c->d_exc.ensure((size_t)(nchunk + 2) * 2));
    CUDA_TRY(c, c->d_key.ensure((size_t)n * 8));
    CUDA_TRY(c, c->d_flags.ensure((size_t)n));
    CUDA_TRY(c, c->d_rep.ensure((size_t)n * 4));
    CUDA_TRY(c, c->d_strand.ensure((size_t)n));
    CUDA_TRY(c, c->d_abund.ensure((size_t)n * 4));
    CUDA_TRY(c, c->d_uid.ensure((size_t)n * 4));
    CUDA_TRY(c, c->d_scan.ensure((size_t)(n + 1) * 4));
    CUDA_TRY(c, c->d_flag.ensure((size_t)(n + 1) * 4));
    int64_t cap = 1024;
    while (cap < 2 * n) cap <<= 1;
    CUDA_TRY(c, c->d_table.ensure((size_t)cap * sizeof(Slot)));
    CUDA_TRY(c, c->d_collide.ensure((size_t)n * 4 + 16));
    CUDA_TRY(c, c->d_counters.ensure(64 * 8));
    const unsigned long long mask = (unsigned long long)cap - 1;
    const unsigned long long keymask = c->key_bits >= 64 ? ~0ull : ((1ull << c->key_bits) - 1ull);

    Timeline<6> tl;     // the ends of pack, hash, insert, verify and compact
    CUDA_TRY(c, tl.status);
    auto *P = c->d_pack2.as<uint32_t>();
    auto *X = c->d_exc.as<uint16_t>();
    auto *ascii = c->d_ascii.as<uint8_t>();
    auto *off = c->d_off.as<int64_t>();
    unsigned long long *d_ncol = c->d_counters.as<unsigned long long>() + CNT_COLLIDE;

    CUDA_TRY(c, tl.record(0, st));
    CUDA_TRY(c, cudaMemsetAsync(P + nchunk, 0, 8, st));
    CUDA_TRY(c, cudaMemsetAsync(X + nchunk, 0, 4, st));
    pack2_kernel<<<nblk(nchunk, 256), 256, 0, st>>>((const uint4 *)ascii, nchunk, P, X);
    CUDA_TRY(c, tl.record(1, st));
    const int32_t *d_samp = c->have_samples ? c->d_sample.as<int32_t>() : nullptr;
    hash_kernel<<<nblk(n, 128), 128, 0, st>>>(ascii, off, P, X, n, keymask, d_samp, c->d_key.as<unsigned long long>(),
                                              c->d_flags.as<uint8_t>());
    CUDA_TRY(c, tl.record(2, st));
    table_init_kernel<<<nblk(cap, 256), 256, 0, st>>>(c->d_table.as<Slot>(), cap);
    insert_kernel<<<nblk(n, 256), 256, 0, st>>>(c->d_key.as<unsigned long long>(), n, c->d_table.as<Slot>(), mask);
    CUDA_TRY(c, tl.record(3, st));
    CUDA_TRY(c, cudaMemsetAsync(c->d_abund.p, 0, (size_t)n * 4, st));
    CUDA_TRY(c, cudaMemsetAsync(d_ncol, 0, 8, st));
    verify_kernel<<<nblk(n, 128), 128, 0, st>>>(ascii, off, P, c->d_key.as<unsigned long long>(),
                                                c->d_flags.as<uint8_t>(), d_samp, n, c->d_table.as<Slot>(), mask,
                                                c->d_rep.as<int32_t>(), c->d_strand.as<uint8_t>(),
                                                c->d_abund.as<int32_t>(), c->d_collide.as<int32_t>(), d_ncol);
    c->launches += 5;
    unsigned long long ncol = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&ncol, d_ncol, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    if (ncol > 0) {
        if (ncol > (1ull << 18)) {
            c->err = "derep: too many 64-bit key collisions to resolve exactly";
            return ITSX_ECOLLIDE;
        }
        collide_kernel<<<nblk((int64_t)ncol, 64), 64, 0, st>>>(ascii, off, P, c->d_flags.as<uint8_t>(), d_samp,
                                                               c->d_collide.as<int32_t>(), (int64_t)ncol,
                                                               c->d_rep.as<int32_t>(), c->d_strand.as<uint8_t>(),
                                                               c->d_abund.as<int32_t>());
        c->launches++;
    }
    ds.n_collided = (int64_t)ncol;
    CUDA_TRY(c, tl.record(4, st));

    // dense ids
    int32_t *flag = c->d_flag.as<int32_t>(), *scan = c->d_scan.as<int32_t>();
    isrep_kernel<<<nblk(n, 256), 256, 0, st>>>(c->d_rep.as<int32_t>(), n, flag);
    CUDA_TRY(c, cudaMemsetAsync(flag + n, 0, 4, st));
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) {
        return cub::DeviceScan::ExclusiveSum(t, b, flag, scan, (int)n + 1, st);
    }));
    int32_t nu = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&nu, scan + n, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    c->n_unique = nu;
    CUDA_TRY(c, c->d_first.ensure((size_t)std::max(nu, 1) * 4));
    first_kernel<<<nblk(n, 256), 256, 0, st>>>(c->d_rep.as<int32_t>(), scan, n, c->d_first.as<int32_t>());
    uid_kernel<<<nblk(n, 256), 256, 0, st>>>(c->d_rep.as<int32_t>(), scan, n, c->d_uid.as<int32_t>());
    c->launches += 5;
    CUDA_TRY(c, tl.record(5, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    ds.ms_pack = tl.ms(0, 1);
    ds.ms_hash = tl.ms(1, 2);
    ds.ms_insert = tl.ms(2, 3);
    ds.ms_verify = tl.ms(3, 4);
    ds.ms_compact = tl.ms(4, 5);
    ds.ms_total = tl.ms(0, 5);
    ds.n_unique = nu;
    c->pos_valid = false;
    c->stage1_done = c->stage2_done = false;
    return ITSX_OK;
}
