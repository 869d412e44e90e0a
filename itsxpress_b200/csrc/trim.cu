// trim.cu -- boundary lookup, keep filter and slice/re-expansion for every input read.
//
// Replaces the per-read Python/Biopython loops of Dedup._get_trimmed_seq_generator
// (itsxpress/SeqSample.py:792-884: filter :814-825, slice :862) and Dedup._get_paired_seq_generator
// (SeqSample.py:564-711: filter :586-598, slices :639-655).  A read is kept iff its representative
// has a left and a right boundary and start < stop; slices follow Python's slice clipping.
// Both kernels are streaming, HBM-bound byte movers: one thread per read for the bounds, one warp per
// kept read for the copy.
#include <cub/cub.cuh>
#include "itsx_internal.h"

namespace {

inline unsigned nblk(int64_t n, int b) { return (unsigned)((n + b - 1) / b); }

// Python's  s[a:b]  on a sequence of length n  ->  [lo, hi)
__device__ __forceinline__ void py_slice(long long a, long long b, long long n, int32_t &lo, int32_t &hi)
{
    if (a < 0) { a += n; if (a < 0) a = 0; }
    if (b < 0) { b += n; if (b < 0) b = 0; }
    if (a > n) a = n;
    if (b > n) b = n;
    if (b < a) b = a;
    lo = (int32_t)a;
    hi = (int32_t)b;
}

__global__ void __launch_bounds__(256)
bounds_kernel(const int32_t *__restrict__ uid, const int32_t *__restrict__ pos, int64_t npos,
              const int64_t *__restrict__ off, int64_t nreads, int mode,
              uint8_t *__restrict__ keep, int32_t *__restrict__ lo, int32_t *__restrict__ hi,
              int32_t *__restrict__ keepflag, int64_t *__restrict__ outlen)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nreads) return;
    const int32_t u = uid[i];
    int32_t k = 0, l = 0, h = 0;
    if (u >= 0 && u < npos) {
        const int32_t start = pos[u], stop = pos[npos + u], tlen = pos[2 * npos + u];
        if (start >= 0 && stop >= 0 && start < stop) {
            k = 1;
            const long long n = off[i + 1] - off[i];
            if (mode == 0) {
                py_slice(start, stop, n, l, h);
            } else if (mode == 2) {
                if (stop > tlen) py_slice(start, n, n, l, h);
                else py_slice(start, stop, n, l, h);
            } else {
                const long long r2start = (long long)tlen - stop, r2end = (long long)tlen - start;
                if (r2end > tlen) py_slice(r2start, n, n, l, h);
                else py_slice(r2start, r2end, n, l, h);
            }
        }
    }
    keep[i] = (uint8_t)k;
    lo[i] = l;
    hi[i] = h;
    if (keepflag) keepflag[i] = k;
    if (outlen) outlen[i] = k ? (int64_t)(h - l) : 0;
}

struct GatherRec { int64_t src, dst; int32_t n, pad; };     // one kept read: where its slice starts, where it goes, how long

__global__ void kept_index_kernel(const int32_t *__restrict__ keepflag, const int32_t *__restrict__ kscan,
                                  const int64_t *__restrict__ lscan, const int64_t *__restrict__ off,
                                  const int32_t *__restrict__ lo, const int32_t *__restrict__ hi, int64_t nreads,
                                  int32_t *__restrict__ kept_index, int64_t *__restrict__ out_off,
                                  GatherRec *__restrict__ rec)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > nreads) return;
    if (i == nreads) { out_off[kscan[nreads]] = lscan[nreads]; return; }
    if (keepflag[i]) {
        const int32_t t = kscan[i];
        kept_index[t] = (int32_t)i;
        out_off[t] = lscan[i];
        GatherRec r;
        r.src = off[i] + lo[i]; r.dst = lscan[i]; r.n = hi[i] - lo[i]; r.pad = 0;
        rec[t] = r;
    }
}

// eight lanes per kept read (trimmed ITS slices are ~130-250 bytes = 8-16 vectors): the seq and qual slices go to the packed
// outputs with 16-byte stores on the aligned middle of the destination (itsx_internal.h: group_copy); one 24-byte record
// per read replaces the five dependent index loads
constexpr int GATHER_W = 8;
__global__ void __launch_bounds__(256)
gather_kernel(const uint8_t *__restrict__ seq, const uint8_t *__restrict__ qual, const GatherRec *__restrict__ rec,
              int64_t nkept, uint8_t *__restrict__ out_seq, uint8_t *__restrict__ out_qual)
{
    const int lane = threadIdx.x & (GATHER_W - 1);
    int64_t t = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / GATHER_W;
    if (t >= nkept) return;
    const GatherRec r = rec[t];
    group_copy(seq + r.src, out_seq + r.dst, r.n, lane, GATHER_W);
    if (qual) group_copy(qual + r.src, out_qual + r.dst, r.n, lane, GATHER_W);
}

}  // namespace

int trim_bounds_dev(itsx_ctx *c, int mode, const int64_t *d_off, int64_t first, int64_t count)
{
    cudaStream_t st = c->stream;
    if (!c->pos_valid) { c->err = "trim: no position table (run itsx_search or itsx_positions_set first)"; return ITSX_EINVAL; }
    if (first < 0 || count < 0 || first + count > c->nreads) {
        c->err = "trim: read range outside the dereplicated set";
        return ITSX_EINVAL;
    }
    c->r_gathered = false;
    c->r_n = count;
    c->r_off = d_off ? d_off : c->d_off.as<int64_t>() + first;
    c->r_nkept = c->r_total = 0;
    CUDA_TRY(c, c->r_keep.ensure((size_t)count + 16));
    CUDA_TRY(c, c->r_lo.ensure((size_t)count * 4 + 16));
    CUDA_TRY(c, c->r_hi.ensure((size_t)count * 4 + 16));
    if (count == 0) return ITSX_OK;
    // keep flags and slice lengths, and their exclusive scans (kept rank, output offset): what trim_gather_dev reads
    CUDA_TRY(c, c->d_flag.ensure((size_t)(count + 1) * 4));
    CUDA_TRY(c, c->d_scan.ensure((size_t)(count + 1) * 4));
    CUDA_TRY(c, c->d_list.ensure((size_t)(count + 1) * 8));
    CUDA_TRY(c, c->d_list2.ensure((size_t)(count + 1) * 8));
    int32_t *kf = c->d_flag.as<int32_t>(), *ks = c->d_scan.as<int32_t>();
    int64_t *ol = c->d_list.as<int64_t>(), *os = c->d_list2.as<int64_t>();
    bounds_kernel<<<nblk(count, 256), 256, 0, st>>>(c->d_uid.as<int32_t>() + first, c->d_pos.as<int32_t>(), c->npos, c->r_off,
                                                    count, mode, c->r_keep.as<uint8_t>(), c->r_lo.as<int32_t>(),
                                                    c->r_hi.as<int32_t>(), kf, ol);
    CUDA_TRY(c, cudaMemsetAsync(kf + count, 0, 4, st));
    CUDA_TRY(c, cudaMemsetAsync(ol + count, 0, 8, st));
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, kf, ks, (int)count + 1, st); },
                        [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, ol, os, (int)count + 1, st); }));
    c->launches += 3;
    int32_t nk = 0;
    int64_t tot = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&nk, ks + count, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaMemcpyAsync(&tot, os + count, 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    c->r_nkept = nk;
    c->r_total = tot;
    return ITSX_OK;
}

int trim_gather_dev(itsx_ctx *c, const uint8_t *d_seq, const uint8_t *d_qual)
{
    cudaStream_t st = c->stream;
    const int64_t n = c->r_n, nk = c->r_nkept, tot = c->r_total;
    CUDA_TRY(c, c->r_ki.ensure((size_t)std::max<int64_t>(nk, 1) * 4));
    CUDA_TRY(c, c->r_oo.ensure((size_t)(nk + 1) * 8));
    CUDA_TRY(c, c->r_os.ensure((size_t)std::max<int64_t>(tot, 1)));
    if (d_qual) CUDA_TRY(c, c->r_oq.ensure((size_t)std::max<int64_t>(tot, 1)));
    if (n == 0) {
        CUDA_TRY(c, cudaMemsetAsync(c->r_oo.p, 0, 8, st));
    } else {
        CUDA_TRY(c, c->d_gather.ensure((size_t)std::max<int64_t>(nk, 1) * sizeof(GatherRec)));
        kept_index_kernel<<<nblk(n + 1, 256), 256, 0, st>>>(c->d_flag.as<int32_t>(), c->d_scan.as<int32_t>(),
                                                            c->d_list2.as<int64_t>(), c->r_off, c->r_lo.as<int32_t>(),
                                                            c->r_hi.as<int32_t>(), n, c->r_ki.as<int32_t>(),
                                                            c->r_oo.as<int64_t>(), c->d_gather.as<GatherRec>());
        if (nk > 0)
            gather_kernel<<<nblk(nk * GATHER_W, 256), 256, 0, st>>>(d_seq, d_qual, c->d_gather.as<GatherRec>(), nk,
                                                                    c->r_os.as<uint8_t>(),
                                                                    d_qual ? c->r_oq.as<uint8_t>() : nullptr);
        c->launches += 2;
        CUDA_TRY(c, cudaGetLastError());
    }
    c->r_gathered = true;
    c->r_gathered_qual = d_qual != nullptr;
    return ITSX_OK;
}

int trim_fetch_dev(itsx_ctx *c, int32_t *kept_index, int64_t *out_off, uint8_t *out_seq, uint8_t *out_qual)
{
    cudaStream_t st = c->stream;
    const int64_t nk = c->r_nkept, tot = c->r_total;
    if (kept_index && nk) CUDA_TRY(c, cudaMemcpyAsync(kept_index, c->r_ki.p, (size_t)nk * 4, cudaMemcpyDefault, st));
    if (out_off) CUDA_TRY(c, cudaMemcpyAsync(out_off, c->r_oo.p, (size_t)(nk + 1) * 8, cudaMemcpyDefault, st));
    if (out_seq && tot) CUDA_TRY(c, cudaMemcpyAsync(out_seq, c->r_os.p, (size_t)tot, cudaMemcpyDefault, st));
    if (out_qual && tot && c->r_gathered_qual) CUDA_TRY(c, cudaMemcpyAsync(out_qual, c->r_oq.p, (size_t)tot, cudaMemcpyDefault, st));
    return ITSX_OK;
}
