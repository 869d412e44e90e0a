// shard.cu -- one sample sharded over the G GPUs of a box: the regrouping kernels on both sides of the
// two exchanges (SURVEY.md 8e).  The exchanges themselves are NCCL collectives issued by the host driver
// (itsxpress_b200/distributed.py) on the buffers these entry points fill / consume.
//
// The reference runs ONE `vsearch --fastx_uniques` and ONE `hmmsearch` per sample (itsxpress/SeqSample.py:106-116,
// 191-209); both are global operations (first occurrence of a class; hmmsearch's per-profile domZ).  Sharded:
//
//   local ctx  (this rank's block of reads, input order)        owner ctx (classes with key64 % G == rank)
//   ------------------------------------------------------      ------------------------------------------------
//   itsx_derep_resident         exact derep of the block
//   itsx_shard_plan             owner of every local unique, stable bucket by owner, G counters -> host
//   itsx_shard_pack             record stream (gidx32 | len32) + bases, grouped by owner
//        ---- all-to-all (records, bases) ---->                  itsx_shard_owner_derep   arrival order = source-rank
//                                                                order = ascending global read index, so the first
//                                                                occurrence of a class is its first arrival; exact
//                                                                derep (every class verified base by base) + search set
//                                                                itsx_search_stage1 / all-reduce domZ / stage2
//        <--- inverse all-to-all (16 B answers) ----             itsx_shard_answers       {rep gidx | strand, start, stop, tlen}
//   itsx_shard_apply            answers -> position table per local unique, global representative per read
//   itsx_trim_bounds / itsx_trim_gather  on the block
//
// No global table is gathered: a rank only learns the positions of the classes its own reads belong to.
#include <cub/cub.cuh>
#include <algorithm>
#include "itsx_internal.h"

namespace {

inline unsigned nblk(int64_t n, int b) { return (unsigned)((n + b - 1) / b); }

// owner rank and length of every local unique; G counters of records and bytes
__global__ void __launch_bounds__(256)
owner_kernel(const unsigned long long *__restrict__ key, const int32_t *__restrict__ first,
             const int64_t *__restrict__ off, int64_t nu, int G, uint8_t *__restrict__ owner,
             int32_t *__restrict__ uidx, unsigned long long *__restrict__ counts)
{
    __shared__ unsigned long long s_cnt[2 * 64];
    for (int t = threadIdx.x; t < 2 * G; t += blockDim.x) s_cnt[t] = 0ull;
    __syncthreads();
    const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < nu) {
        const int32_t r = first[u];
        const int o = (int)(key[r] % (unsigned long long)G);
        owner[u] = (uint8_t)o;
        uidx[u] = (int32_t)u;
        atomicAdd(&s_cnt[o], 1ull);
        atomicAdd(&s_cnt[G + o], (unsigned long long)(off[r + 1] - off[r]));
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * G; t += blockDim.x)
        if (s_cnt[t]) atomicAdd(&counts[t], s_cnt[t]);
}

// record stream in bucket order + the length of every record (input of the byte-offset scan)
__global__ void __launch_bounds__(256)
record_kernel(const int32_t *__restrict__ order, const int32_t *__restrict__ first, const int64_t *__restrict__ off,
              int64_t nu, int64_t gidx0, unsigned long long *__restrict__ rec, int64_t *__restrict__ len64)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j > nu) return;
    if (j == nu) { len64[j] = 0; return; }
    const int32_t r = first[order[j]];
    const int64_t L = off[r + 1] - off[r];
    rec[j] = (unsigned long long)(gidx0 + r) | ((unsigned long long)L << 32);
    len64[j] = L;
}

__global__ void __launch_bounds__(256)
pack_bases_kernel(const uint8_t *__restrict__ ascii, const int64_t *__restrict__ off, const int32_t *__restrict__ order,
                  const int32_t *__restrict__ first, const int64_t *__restrict__ doff, int64_t nu,
                  uint8_t *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (j >= nu) return;
    const int32_t r = first[order[j]];
    const int64_t s = off[r];
    warp_copy(ascii + s, out + doff[j], (int)(off[r + 1] - s), lane);
}

__global__ void reclen_kernel(const unsigned long long *__restrict__ rec, int64_t n, int64_t *__restrict__ len64)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j > n) return;
    len64[j] = j < n ? (int64_t)(rec[j] >> 32) : 0;
}

// owner side: one 16-byte answer per received record
__global__ void __launch_bounds__(256)
answer_kernel(const unsigned long long *__restrict__ rec, const int32_t *__restrict__ rep,
              const uint8_t *__restrict__ strand, const int32_t *__restrict__ uid, const int32_t *__restrict__ pos,
              int64_t npos, int64_t n, int4 *__restrict__ ans)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t g = (uint32_t)(rec[rep[j]] & 0xffffffffull);
    const int32_t u = uid[j];
    int4 a;
    a.x = (int32_t)(g | ((uint32_t)(strand[j] & 1) << 31));
    a.y = pos[u]; a.z = pos[npos + u]; a.w = pos[2 * npos + u];
    ans[j] = a;
}

// local side: answers (bucket order) -> per local unique
__global__ void __launch_bounds__(256)
apply_unique_kernel(const int4 *__restrict__ ans, const int32_t *__restrict__ order, int64_t nu,
                    int32_t *__restrict__ pos, int32_t *__restrict__ repg)
{
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nu) return;
    const int4 a = ans[j];
    const int32_t u = order[j];
    pos[u] = a.y; pos[nu + u] = a.z; pos[2 * nu + u] = a.w;
    repg[u] = a.x;
}
__global__ void __launch_bounds__(256)
apply_read_kernel(const int32_t *__restrict__ uid, const int32_t *__restrict__ repg, const uint8_t *__restrict__ strand_l,
                  int64_t n, int64_t *__restrict__ rep_global, uint8_t *__restrict__ strand)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t g = (uint32_t)repg[uid[i]];
    if (rep_global) rep_global[i] = (int64_t)(g & 0x7fffffffu);
    if (strand) strand[i] = (uint8_t)((strand_l[i] ^ (g >> 31)) & 1u);
}

}  // namespace

#define CHECK_CTX(c) do { if (!(c)) return ITSX_EINVAL; } while (0)

extern "C" {

int itsx_derep_resident(itsx_ctx *c, int build_search_set, int64_t *n_unique)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (c->map_external) { c->err = "derep_resident: no reads are resident (itsx_reads_upload first)"; return ITSX_EINVAL; }
    int rc = derep_run(c);
    if (rc) return rc;
    if (n_unique) *n_unique = c->n_unique;
    c->shard_first = 0;
    c->shard_n = -1;
    c->sh_G = 0;
    if (build_search_set) return search_build_seqs_from_derep(c);
    return ITSX_OK;
}

int itsx_shard_plan(itsx_ctx *c, int G, int64_t *rec_counts, int64_t *byte_counts)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (G < 1 || G > 64) { c->err = "shard_plan: G must be 1..64"; return ITSX_EINVAL; }
    if (c->map_external || c->dstats.n_reads != c->nreads) { c->err = "shard_plan: run itsx_derep on the block first"; return ITSX_EINVAL; }
    cudaStream_t st = c->stream;
    const int64_t nu = c->n_unique;
    c->sh_G = G;
    CUDA_TRY(c, c->d_counters.ensure(64 * 8 + 2 * 64 * 8));
    unsigned long long *d_cnt = c->d_counters.as<unsigned long long>() + 64;
    CUDA_TRY(c, cudaMemsetAsync(d_cnt, 0, 2 * 64 * 8, st));
    CUDA_TRY(c, c->d_sh_order.ensure((size_t)std::max<int64_t>(nu, 1) * 4));
    if (nu > 0) {
        // scratch: owner (u8) in / out, identity index in
        const size_t idx_at = ((size_t)2 * nu + 15) & ~(size_t)15;
        CUDA_TRY(c, c->d_sh_tmp.ensure(idx_at + (size_t)nu * 4));
        uint8_t *own_in = c->d_sh_tmp.as<uint8_t>(), *own_out = own_in + nu;
        int32_t *idx_in = (int32_t *)(c->d_sh_tmp.as<uint8_t>() + idx_at);
        owner_kernel<<<nblk(nu, 256), 256, 0, st>>>(c->d_key.as<unsigned long long>(), c->d_first.as<int32_t>(),
                                                    c->d_off.as<int64_t>(), nu, G, own_in, idx_in, d_cnt);
        int bits = 1;
        while ((1 << bits) < G) bits++;
        // stable: inside a bucket the uniques stay in first-occurrence order = ascending global read index
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) {
            return cub::DeviceRadixSort::SortPairs(t, b, own_in, own_out, idx_in, c->d_sh_order.as<int32_t>(), (int)nu, 0, bits, st);
        }));
        c->launches += 2;
    }
    unsigned long long h[2 * 64];
    CUDA_TRY(c, cudaMemcpyAsync(h, d_cnt, sizeof(h), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    c->sh_bytes = 0;
    for (int g = 0; g < G; g++) {
        if (rec_counts) rec_counts[g] = (int64_t)h[g];
        if (byte_counts) byte_counts[g] = (int64_t)h[G + g];
        c->sh_bytes += (int64_t)h[G + g];
    }
    return ITSX_OK;
}

int itsx_shard_pack(itsx_ctx *c, int64_t first_global_index, uint64_t *rec, uint8_t *bases)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (c->sh_G < 1) { c->err = "shard_pack before shard_plan"; return ITSX_EINVAL; }
    const int64_t nu = c->n_unique;
    if (first_global_index < 0 || first_global_index + c->nreads > 0x7fffffffLL) {
        c->err = "shard_pack: global read indices must stay below 2^31";
        return ITSX_ELIMIT;
    }
    if (nu == 0) return ITSX_OK;
    if (!rec || (!bases && c->sh_bytes)) { c->err = "shard_pack: null buffer"; return ITSX_EINVAL; }
    cudaStream_t st = c->stream;
    // records and bases are produced in library scratch, then copied to the caller's buffers (host or device)
    CUDA_TRY(c, c->d_sh_tmp.ensure((size_t)(nu + 1) * 8 * 3 + 64));
    unsigned long long *d_rec = c->d_sh_tmp.as<unsigned long long>();
    int64_t *d_len = (int64_t *)(d_rec + (nu + 1)), *d_doff = d_len + (nu + 1);
    CUDA_TRY(c, c->d_sh_bases.ensure((size_t)c->sh_bytes + 64));
    record_kernel<<<nblk(nu + 1, 256), 256, 0, st>>>(c->d_sh_order.as<int32_t>(), c->d_first.as<int32_t>(),
                                                     c->d_off.as<int64_t>(), nu, first_global_index, d_rec, d_len);
    CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) { return cub::DeviceScan::ExclusiveSum(t, b, d_len, d_doff, (int)nu + 1, st); }));
    pack_bases_kernel<<<nblk(nu * 32, 256), 256, 0, st>>>(c->d_ascii.as<uint8_t>(), c->d_off.as<int64_t>(),
                                                          c->d_sh_order.as<int32_t>(), c->d_first.as<int32_t>(), d_doff,
                                                          nu, c->d_sh_bases.as<uint8_t>());
    c->launches += 3;
    CUDA_TRY(c, cudaMemcpyAsync(rec, d_rec, (size_t)nu * 8, cudaMemcpyDefault, st));
    if (c->sh_bytes) CUDA_TRY(c, cudaMemcpyAsync(bases, c->d_sh_bases.p, (size_t)c->sh_bytes, cudaMemcpyDefault, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    return ITSX_OK;
}

int itsx_shard_owner_derep(itsx_ctx *c, const uint64_t *rec, int64_t nrec, const uint8_t *bases, int64_t nbytes,
                           int64_t *n_own)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (nrec < 0 || nbytes < 0 || (nrec && !rec) || (nbytes && !bases)) { c->err = "shard_owner_derep: bad argument"; return ITSX_EINVAL; }
    cudaStream_t st = c->stream;
    reset_reads(c, nrec, nbytes);
    c->sh_G = 0;
    const size_t padded = ((size_t)nbytes + 15) / 16 * 16 + 32;
    CUDA_TRY(c, c->d_ascii.ensure(padded));
    CUDA_TRY(c, c->d_off.ensure((size_t)(nrec + 1) * 8));
    CUDA_TRY(c, c->d_sh_rec.ensure((size_t)std::max<int64_t>(nrec, 1) * 8));
    CUDA_TRY(c, cudaMemsetAsync(c->d_ascii.as<uint8_t>() + (size_t)nbytes / 16 * 16, 'A', padded - (size_t)nbytes / 16 * 16, st));
    if (nbytes) CUDA_TRY(c, cudaMemcpyAsync(c->d_ascii.p, bases, (size_t)nbytes, cudaMemcpyDefault, st));
    if (nrec) {
        CUDA_TRY(c, cudaMemcpyAsync(c->d_sh_rec.p, rec, (size_t)nrec * 8, cudaMemcpyDefault, st));
        CUDA_TRY(c, c->d_sh_tmp.ensure((size_t)(nrec + 1) * 8));
        int64_t *d_len = c->d_sh_tmp.as<int64_t>();
        reclen_kernel<<<nblk(nrec + 1, 256), 256, 0, st>>>(c->d_sh_rec.as<unsigned long long>(), nrec, d_len);
        CUDA_TRY(c, cub_run(c, [&](void *t, size_t &b) {
            return cub::DeviceScan::ExclusiveSum(t, b, d_len, c->d_off.as<int64_t>(), (int)nrec + 1, st);
        }));
        c->launches += 2;
        int64_t tot = 0;
        CUDA_TRY(c, cudaMemcpyAsync(&tot, c->d_off.as<int64_t>() + nrec, 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        if (tot != nbytes) { c->err = "shard_owner_derep: record lengths do not add up to the byte count"; return ITSX_EINVAL; }
    } else {
        CUDA_TRY(c, cudaMemsetAsync(c->d_off.p, 0, 8, st));
    }
    int rc = derep_run(c);
    if (rc) return rc;
    if (n_own) *n_own = c->n_unique;
    c->shard_first = 0;
    c->shard_n = -1;
    return search_build_seqs_from_derep(c);
}

int itsx_shard_answers(itsx_ctx *c, int64_t nrec, int32_t *ans)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (nrec != c->nreads) { c->err = "shard_answers: record count differs from the owner's read set"; return ITSX_EINVAL; }
    if (nrec == 0) return ITSX_OK;
    if (!c->pos_valid || c->npos != c->n_unique) { c->err = "shard_answers before the search finished"; return ITSX_EINVAL; }
    if (!ans) return ITSX_EINVAL;
    cudaStream_t st = c->stream;
    CUDA_TRY(c, c->d_sh_tmp.ensure((size_t)nrec * 16));
    answer_kernel<<<nblk(nrec, 256), 256, 0, st>>>(c->d_sh_rec.as<unsigned long long>(), c->d_rep.as<int32_t>(),
                                                   c->d_strand.as<uint8_t>(), c->d_uid.as<int32_t>(),
                                                   c->d_pos.as<int32_t>(), c->npos, nrec, c->d_sh_tmp.as<int4>());
    c->launches++;
    CUDA_TRY(c, cudaMemcpyAsync(ans, c->d_sh_tmp.p, (size_t)nrec * 16, cudaMemcpyDefault, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    return ITSX_OK;
}

int itsx_shard_apply(itsx_ctx *c, const int32_t *ans, int64_t nu, int64_t *rep_global, uint8_t *strand)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (c->sh_G < 1) { c->err = "shard_apply before shard_plan"; return ITSX_EINVAL; }
    if (nu != c->n_unique) { c->err = "shard_apply: answer count differs from the block's unique count"; return ITSX_EINVAL; }
    cudaStream_t st = c->stream;
    const int64_t n = c->nreads;
    c->npos = nu;
    CUDA_TRY(c, c->d_pos.ensure((size_t)std::max<int64_t>(nu, 1) * 9 * 4));
    if (nu) {
        if (!ans) return ITSX_EINVAL;
        const size_t rg_at = ((size_t)nu * 20 + 15) & ~(size_t)15;
        CUDA_TRY(c, c->d_sh_tmp.ensure(rg_at + (size_t)n * 9 + 64));
        int4 *d_ans = c->d_sh_tmp.as<int4>();
        int32_t *d_repg = (int32_t *)(d_ans + nu);
        int64_t *d_rg = (int64_t *)(c->d_sh_tmp.as<char>() + rg_at);
        uint8_t *d_st = (uint8_t *)(d_rg + n);
        CUDA_TRY(c, cudaMemcpyAsync(d_ans, ans, (size_t)nu * 16, cudaMemcpyDefault, st));
        CUDA_TRY(c, cudaMemsetAsync(c->d_pos.p, 0xff, (size_t)nu * 9 * 4, st));
        apply_unique_kernel<<<nblk(nu, 256), 256, 0, st>>>(d_ans, c->d_sh_order.as<int32_t>(), nu, c->d_pos.as<int32_t>(), d_repg);
        c->launches++;
        if (n && (rep_global || strand)) {
            apply_read_kernel<<<nblk(n, 256), 256, 0, st>>>(c->d_uid.as<int32_t>(), d_repg, c->d_strand.as<uint8_t>(), n,
                                                            rep_global ? d_rg : nullptr, strand ? d_st : nullptr);
            c->launches++;
            if (rep_global) CUDA_TRY(c, cudaMemcpyAsync(rep_global, d_rg, (size_t)n * 8, cudaMemcpyDefault, st));
            if (strand) CUDA_TRY(c, cudaMemcpyAsync(strand, d_st, (size_t)n, cudaMemcpyDefault, st));
        }
    }
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    c->pos_valid = true;
    return ITSX_OK;
}

}  // extern "C"
