// api.cu -- the extern "C" surface of libitsx_b200.so (declared in include/itsx_b200.h): context,
// profile loading, host<->device staging and the glue between the stage implementations in
// derep.cu / search.cu / trim.cu.  No compute happens on the host: a missing or non-sm_100 device
// makes itsx_create fail (there is no CPU fallback).
#include <algorithm>
#include <cstring>
#include <numeric>
#include "itsx_internal.h"

static thread_local std::string g_create_err;

DevBuf::~DevBuf()
{
    if (p) cudaFree(p);
}
cudaError_t DevBuf::ensure(size_t bytes, bool keep, cudaStream_t st)
{
    if (bytes <= cap && p) return cudaSuccess;
    size_t ncap = std::max(bytes, cap + cap / 2);
    ncap = (ncap + 255) & ~(size_t)255;
    void *q = nullptr;
    cudaError_t e = cudaMalloc(&q, ncap);
    if (e != cudaSuccess) return e;
    if (p) {
        if (keep && cap) {
            e = cudaMemcpyAsync(q, p, cap, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) { cudaFree(q); return e; }
        }
        cudaFree(p);
    }
    p = q;
    cap = ncap;
    return cudaSuccess;
}

#define CHECK_CTX(c) do { if (!(c)) return ITSX_EINVAL; } while (0)

extern "C" {

int itsx_create(int device, itsx_ctx **out)
{
    if (!out) return ITSX_EINVAL;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_err = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return ITSX_ENODEV;
    }
    if (device < 0 || device >= ndev) { g_create_err = "device index out of range"; return ITSX_EINVAL; }
    cudaDeviceProp pr;
    if ((e = cudaGetDeviceProperties(&pr, device)) != cudaSuccess) { g_create_err = cudaGetErrorString(e); return ITSX_ECUDA; }
    if (pr.major != 10) {
        g_create_err = "libitsx_b200 is built for sm_100a only; device is sm_" + std::to_string(pr.major * 10 + pr.minor);
        return ITSX_ENODEV;
    }
    if ((e = cudaSetDevice(device)) != cudaSuccess) { g_create_err = cudaGetErrorString(e); return ITSX_ECUDA; }
    itsx_ctx *c = new itsx_ctx();
    c->device = device;
    c->sm_count = pr.multiProcessorCount;
    c->cc_major = pr.major;
    c->cc_minor = pr.minor;
    c->mem_total = pr.totalGlobalMem;
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        g_create_err = cudaGetErrorString(e);
        delete c;
        return ITSX_ECUDA;
    }
    itsx_search_default_params(&c->prm);
    *out = c;
    return ITSX_OK;
}

void itsx_destroy(itsx_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (auto s : c->lanes) cudaStreamDestroy(s);
    for (auto e : c->lane_ev) cudaEventDestroy(e);
    if (c->lane_fork) cudaEventDestroy(c->lane_fork);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

const char *itsx_last_error(const itsx_ctx *c) { return c ? c->err.c_str() : g_create_err.c_str(); }

int itsx_device_info(const itsx_ctx *c, int *sm_count, int *cc_major, int *cc_minor, int64_t *mem_bytes)
{
    CHECK_CTX(c);
    if (sm_count) *sm_count = c->sm_count;
    if (cc_major) *cc_major = c->cc_major;
    if (cc_minor) *cc_minor = c->cc_minor;
    if (mem_bytes) *mem_bytes = (int64_t)c->mem_total;
    return ITSX_OK;
}
void *itsx_stream(const itsx_ctx *c) { return c ? (void *)c->stream : nullptr; }
int itsx_sync(itsx_ctx *c)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ITSX_OK;
}
int64_t itsx_launch_count(const itsx_ctx *c) { return c ? c->launches : 0; }

void *itsx_pinned_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void itsx_pinned_free(void *p)
{
    if (p) cudaFreeHost(p);
}

// ---- profiles -------------------------------------------------------------------------------
int itsx_profiles_clear(itsx_ctx *c)
{
    CHECK_CTX(c);
    c->prof.clear();
    c->side.clear();
    c->prof_dirty = true;
    return ITSX_OK;
}
int itsx_profiles_append_file(itsx_ctx *c, const char *path, const char *const *prefixes, int nprefix)
{
    CHECK_CTX(c);
    if (!path) return ITSX_EINVAL;
    int n = hmmfile_append(path, prefixes, nprefix, c->prof, c->err);
    if (n < 0) return n;
    for (size_t p = c->prof.size() - n; p < c->prof.size(); p++)
        if (c->prof[p].M > ITSX_MAXM) {
            c->err = "profile '" + c->prof[p].name + "' is longer than ITSX_MAXM";
            c->prof.resize(c->prof.size() - n);
            return ITSX_ELIMIT;
        }
    c->side.resize(c->prof.size(), -1);
    c->prof_dirty = true;
    return n;
}
int itsx_profiles_count(const itsx_ctx *c) { return c ? (int)c->prof.size() : 0; }
const char *itsx_profile_name(const itsx_ctx *c, int p)
{
    return (c && p >= 0 && p < (int)c->prof.size()) ? c->prof[p].name.c_str() : nullptr;
}
int itsx_profile_M(const itsx_ctx *c, int p) { return (c && p >= 0 && p < (int)c->prof.size()) ? c->prof[p].M : -1; }
int itsx_profiles_set_sides(itsx_ctx *c, const int8_t *side, int n)
{
    CHECK_CTX(c);
    if (n != (int)c->prof.size()) { c->err = "set_sides: length differs from the profile count"; return ITSX_EINVAL; }
    c->side.assign(side, side + n);
    c->prof_dirty = true;
    return ITSX_OK;
}
int itsx_profile_msv(const itsx_ctx *c, int p, uint8_t *cost, int32_t *sc)
{
    CHECK_CTX(c);
    if (p < 0 || p >= (int)c->prof.size()) return ITSX_EINVAL;
    const HostProfile &h = c->prof[p];
    if (cost) memcpy(cost, h.cost.data(), h.cost.size());
    if (sc) { sc[0] = h.bias_b; sc[1] = h.base_b; sc[2] = h.tbm_b; sc[3] = h.tec_b; }
    return ITSX_OK;
}

// ---- reads / derep ---------------------------------------------------------------------------
int itsx_reads_upload(itsx_ctx *c, const uint8_t *seq, const int64_t *off, int64_t nreads)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (nreads < 0 || (nreads > 0 && (!seq || !off))) { c->err = "reads_upload: null buffer"; return ITSX_EINVAL; }
    const int64_t total = nreads ? itsx_peek_i64(off + nreads) : 0;
    if (nreads && itsx_peek_i64(off) != 0) { c->err = "reads_upload: off[0] must be 0"; return ITSX_EINVAL; }
    c->nreads = nreads;
    c->total_bases = total;
    c->n_unique = 0;
    c->cl_active = false;
    c->map_external = false;
    c->pos_valid = false;
    c->qual_resident = false;
    c->r_gathered = false;
    c->have_samples = false;
    c->n_samples = 1;
    c->stream_open = false;
    const size_t padded = ((size_t)total + 15) / 16 * 16 + 32;
    CUDA_TRY(c, c->d_ascii.ensure(padded));
    CUDA_TRY(c, c->d_off.ensure((size_t)(nreads + 1) * 8));
    CUDA_TRY(c, cudaMemsetAsync(c->d_ascii.as<uint8_t>() + (size_t)total / 16 * 16, 'A', padded - (size_t)total / 16 * 16, c->stream));
    if (total) CUDA_TRY(c, cudaMemcpyAsync(c->d_ascii.p, seq, (size_t)total, cudaMemcpyDefault, c->stream));
    if (nreads) CUDA_TRY(c, cudaMemcpyAsync(c->d_off.p, off, (size_t)(nreads + 1) * 8, cudaMemcpyDefault, c->stream));
    else CUDA_TRY(c, cudaMemsetAsync(c->d_off.p, 0, 8, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ITSX_OK;
}

int itsx_reads_set_samples(itsx_ctx *c, const int32_t *sample_of_read, int32_t n_samples)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (c->map_external) { c->err = "reads_set_samples: no reads are resident (itsx_reads_upload first)"; return ITSX_EINVAL; }
    if (n_samples < 1 || (c->nreads && !sample_of_read)) { c->err = "reads_set_samples: bad argument"; return ITSX_EINVAL; }
    CUDA_TRY(c, c->d_sample.ensure((size_t)std::max<int64_t>(c->nreads, 1) * 4));
    if (c->nreads) CUDA_TRY(c, cudaMemcpyAsync(c->d_sample.p, sample_of_read, (size_t)c->nreads * 4, cudaMemcpyDefault, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    c->n_samples = n_samples;
    c->have_samples = true;
    return ITSX_OK;
}

// ---- streamed upload: a file too large to parse in one piece arrives in chunks ------------------------------------
__global__ void offset_append_kernel(const int64_t *__restrict__ chunk_off, int64_t n, int64_t base, int64_t *__restrict__ out)
{
    int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j <= n) out[j] = chunk_off[j] + base;
}

int itsx_reads_begin(itsx_ctx *c, int64_t nreads_hint, int64_t bases_hint)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    c->nreads = 0;
    c->total_bases = 0;
    c->n_unique = 0;
    c->cl_active = false;
    c->map_external = false;
    c->pos_valid = false;
    c->qual_resident = false;
    c->r_gathered = false;
    c->have_samples = false;
    c->n_samples = 1;
    c->stream_open = true;
    c->stream_qual = true;
    c->stream_reads = c->stream_bases = 0;
    CUDA_TRY(c, c->d_ascii.ensure((size_t)std::max<int64_t>(bases_hint, 1 << 20) + 64));
    CUDA_TRY(c, c->d_qual.ensure((size_t)std::max<int64_t>(bases_hint, 1 << 20) + 64));
    CUDA_TRY(c, c->d_off.ensure((size_t)(std::max<int64_t>(nreads_hint, 1024) + 1) * 8));
    CUDA_TRY(c, cudaMemsetAsync(c->d_off.p, 0, 8, c->stream));
    return ITSX_OK;
}

int itsx_reads_append(itsx_ctx *c, const uint8_t *seq, const uint8_t *qual, const int64_t *off, int64_t nreads)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (!c->stream_open) { c->err = "reads_append without itsx_reads_begin"; return ITSX_EINVAL; }
    if (nreads < 0 || (nreads && (!seq || !off))) { c->err = "reads_append: null buffer"; return ITSX_EINVAL; }
    if (nreads == 0) return ITSX_OK;
    if (itsx_peek_i64(off) != 0) { c->err = "reads_append: the chunk's off[0] must be 0"; return ITSX_EINVAL; }
    const int64_t nb = itsx_peek_i64(off + nreads);
    cudaStream_t st = c->stream;
    if (c->stream_reads + nreads >= 0x7fffffffLL) { c->err = "reads_append: more than 2^31-1 reads"; return ITSX_ELIMIT; }
    // (DevBuf grows geometrically and keeps what is there)
    CUDA_TRY(c, c->d_ascii.ensure((size_t)(c->stream_bases + nb) + 64, true, st));
    CUDA_TRY(c, c->d_off.ensure((size_t)(c->stream_reads + nreads + 1) * 8, true, st));
    static thread_local DevBuf t_off;
    CUDA_TRY(c, t_off.ensure((size_t)(nreads + 1) * 8));
    CUDA_TRY(c, cudaMemcpyAsync(c->d_ascii.as<uint8_t>() + c->stream_bases, seq, (size_t)nb, cudaMemcpyDefault, st));
    if (qual && c->stream_qual) {
        CUDA_TRY(c, c->d_qual.ensure((size_t)(c->stream_bases + nb) + 64, true, st));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_qual.as<uint8_t>() + c->stream_bases, qual, (size_t)nb, cudaMemcpyDefault, st));
    } else {
        c->stream_qual = false;
    }
    CUDA_TRY(c, cudaMemcpyAsync(t_off.p, off, (size_t)(nreads + 1) * 8, cudaMemcpyDefault, st));
    offset_append_kernel<<<(unsigned)((nreads + 256) / 256), 256, 0, st>>>(t_off.as<int64_t>(), nreads, c->stream_bases,
                                                                           c->d_off.as<int64_t>() + c->stream_reads);
    c->launches++;
    c->stream_reads += nreads;
    c->stream_bases += nb;
    // the staging copy of the offsets is reused by the next append: drain here (the caller's seq / qual buffers are then
    // free as well; a double-buffering reader fills its OTHER buffer while this call runs on a worker thread)
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return ITSX_OK;
}

int itsx_reads_end(itsx_ctx *c, int64_t *nreads, int64_t *total_bases)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (!c->stream_open) { c->err = "reads_end without itsx_reads_begin"; return ITSX_EINVAL; }
    cudaStream_t st = c->stream;
    const int64_t total = c->stream_bases;
    const size_t padded = ((size_t)total + 15) / 16 * 16 + 32;
    CUDA_TRY(c, c->d_ascii.ensure(padded, true, st));
    CUDA_TRY(c, cudaMemsetAsync(c->d_ascii.as<uint8_t>() + total, 'A', padded - (size_t)total, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    c->nreads = c->stream_reads;
    c->total_bases = total;
    c->qual_resident = c->stream_qual && c->stream_reads > 0;
    c->stream_open = false;
    if (nreads) *nreads = c->nreads;
    if (total_bases) *total_bases = total;
    return ITSX_OK;
}

/* re-expansion of the resident reads [first, first + count): what a chunked writer asks for, chunk after chunk */
int itsx_trim_gather_range(itsx_ctx *c, int mode, int64_t first, int64_t count, int64_t *n_kept, int64_t *total,
                           int32_t *kept_index, int64_t *out_off, uint8_t *out_seq, uint8_t *out_qual)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (c->stream_open) { c->err = "trim: a streamed upload is still open (itsx_reads_end)"; return ITSX_EINVAL; }
    if (mode != 0) { c->err = "trim_gather_range: only mode 0 (the dereplicated reads themselves)"; return ITSX_EINVAL; }
    if (c->map_external) { c->err = "trim_gather_range: no reads are resident"; return ITSX_EINVAL; }
    if (c->npos != map_rows(c)) { c->err = "trim: position table does not cover every unique sequence"; return ITSX_EINVAL; }
    if (first < 0 || count < 0 || first + count > c->nreads) { c->err = "trim_gather_range: range outside the reads"; return ITSX_EINVAL; }
    if (!n_kept || !total) return ITSX_EINVAL;
    cudaStream_t st = c->stream;
    CUDA_TRY(c, c->r_keep.ensure((size_t)count + 16));
    CUDA_TRY(c, c->r_lo.ensure((size_t)count * 4 + 16));
    CUDA_TRY(c, c->r_hi.ensure((size_t)count * 4 + 16));
    int64_t nk = 0;
    int rc = trim_bounds_dev(c, 0, nullptr, count, c->r_keep.as<uint8_t>(), c->r_lo.as<int32_t>(), c->r_hi.as<int32_t>(), &nk,
                             first);
    if (rc) return rc;
    rc = trim_gather_dev(c, c->d_ascii.as<uint8_t>(), c->qual_resident ? c->d_qual.as<uint8_t>() : nullptr,
                         c->d_off.as<int64_t>() + first, count, c->r_keep.as<uint8_t>(), c->r_lo.as<int32_t>(),
                         c->r_hi.as<int32_t>(), n_kept, total, c->r_ki, c->r_oo, c->r_os, c->r_oq);
    if (rc) return rc;
    c->r_gathered = false;
    if (kept_index && *n_kept) CUDA_TRY(c, cudaMemcpyAsync(kept_index, c->r_ki.p, (size_t)*n_kept * 4, cudaMemcpyDefault, st));
    if (out_off) CUDA_TRY(c, cudaMemcpyAsync(out_off, c->r_oo.p, (size_t)(*n_kept + 1) * 8, cudaMemcpyDefault, st));
    if (out_seq && *total) CUDA_TRY(c, cudaMemcpyAsync(out_seq, c->r_os.p, (size_t)*total, cudaMemcpyDefault, st));
    if (out_qual && *total && c->qual_resident) CUDA_TRY(c, cudaMemcpyAsync(out_qual, c->r_oq.p, (size_t)*total, cudaMemcpyDefault, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return ITSX_OK;
}

int itsx_derep(itsx_ctx *c, const uint8_t *seq, const int64_t *off, int64_t nreads,
               int32_t *rep_index, uint8_t *strand, int64_t *n_unique)
{
    CHECK_CTX(c);
    int rc = itsx_reads_upload(c, seq, off, nreads);
    if (rc) return rc;
    rc = derep_run(c);
    if (rc) return rc;
    if (nreads) {
        if (rep_index) CUDA_TRY(c, cudaMemcpyAsync(rep_index, c->d_rep.p, (size_t)nreads * 4, cudaMemcpyDefault, c->stream));
        if (strand) CUDA_TRY(c, cudaMemcpyAsync(strand, c->d_strand.p, (size_t)nreads, cudaMemcpyDefault, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    if (n_unique) *n_unique = c->n_unique;
    // the representatives become the search set
    c->shard_first = 0;
    c->shard_n = -1;
    return search_build_seqs_from_derep(c);
}

__global__ void abund_gather_kernel(const int32_t *__restrict__ first, const int32_t *__restrict__ abund_by_read,
                                    int64_t nu, int32_t *__restrict__ out)
{
    int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < nu) out[u] = abund_by_read[first[u]];
}

int itsx_derep_clusters(itsx_ctx *c, int32_t *first_read, int32_t *abundance)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    const int64_t nu = c->n_unique;
    if (nu == 0) return ITSX_OK;
    if (first_read) CUDA_TRY(c, cudaMemcpyAsync(first_read, c->d_first.p, (size_t)nu * 4, cudaMemcpyDefault, c->stream));
    if (abundance) {
        CUDA_TRY(c, c->d_list.ensure((size_t)nu * 4));
        abund_gather_kernel<<<(unsigned)((nu + 255) / 256), 256, 0, c->stream>>>(c->d_first.as<int32_t>(), c->d_abund.as<int32_t>(), nu,
                                                                                  c->d_list.as<int32_t>());
        c->launches++;
        CUDA_TRY(c, cudaMemcpyAsync(abundance, c->d_list.p, (size_t)nu * 4, cudaMemcpyDefault, c->stream));
    }
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ITSX_OK;
}
__global__ void key_gather_kernel(const int32_t *__restrict__ first, const unsigned long long *__restrict__ key,
                                  int64_t nu, unsigned long long *__restrict__ out)
{
    int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < nu) out[u] = key[first[u]];
}

int itsx_derep_unique_keys(itsx_ctx *c, uint64_t *keys)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    const int64_t nu = c->n_unique;
    if (nu == 0 || !keys) return ITSX_OK;
    if (c->map_external) { c->err = "derep_unique_keys: no dereplicated reads are resident"; return ITSX_EINVAL; }
    CUDA_TRY(c, c->d_list.ensure((size_t)nu * 8));
    key_gather_kernel<<<(unsigned)((nu + 255) / 256), 256, 0, c->stream>>>(c->d_first.as<int32_t>(),
                                                                            c->d_key.as<unsigned long long>(), nu,
                                                                            c->d_list.as<unsigned long long>());
    c->launches++;
    CUDA_TRY(c, cudaMemcpyAsync(keys, c->d_list.p, (size_t)nu * 8, cudaMemcpyDefault, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ITSX_OK;
}

int itsx_derep_map(itsx_ctx *c, int32_t *rep_index, uint8_t *strand, int32_t *uid)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (c->map_external || c->dstats.n_reads != c->nreads) { c->err = "derep_map: no dereplicated reads are resident"; return ITSX_EINVAL; }
    const int64_t n = c->nreads;
    if (n == 0) return ITSX_OK;
    if (rep_index) CUDA_TRY(c, cudaMemcpyAsync(rep_index, c->d_rep.p, (size_t)n * 4, cudaMemcpyDefault, c->stream));
    if (strand) CUDA_TRY(c, cudaMemcpyAsync(strand, c->d_strand.p, (size_t)n, cudaMemcpyDefault, c->stream));
    if (uid) CUDA_TRY(c, cudaMemcpyAsync(uid, c->d_uid.p, (size_t)n * 4, cudaMemcpyDefault, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ITSX_OK;
}

int itsx_derep_get_stats(const itsx_ctx *c, itsx_derep_stats *st)
{
    CHECK_CTX(c);
    if (st) *st = c->dstats;
    return ITSX_OK;
}
int itsx_derep_set_key_bits(itsx_ctx *c, int bits)
{
    CHECK_CTX(c);
    if (bits < 1 || bits > 64) return ITSX_EINVAL;
    c->key_bits = bits;
    return ITSX_OK;
}

// ---- clustering below 100 % identity (cluster.cu; replaces vsearch --cluster_size, SeqSample.py:133-176) --------------
int itsx_cluster(itsx_ctx *c, const itsx_cluster_params *prm, const int32_t *order, int64_t *n_centroids)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    return cluster_run(c, prm, order, n_centroids);
}

int itsx_cluster_set_key_bits(itsx_ctx *c, int bits)
{
    CHECK_CTX(c);
    if (bits < 1 || bits > 64) return ITSX_EINVAL;
    c->cl_key_bits = bits;
    return ITSX_OK;
}

int itsx_cluster_fetch(itsx_ctx *c, int32_t *centroid_row_of_unique, uint8_t *strand_of_unique, int32_t *ed_of_unique,
                       int32_t *unique_of_row)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (!c->cl_active) { c->err = "cluster_fetch: no clustering of the resident derep (itsx_cluster first)"; return ITSX_EINVAL; }
    const int64_t nu = c->n_unique, nc = c->cl_ncent;
    cudaStream_t st = c->stream;
    const int32_t *crow = c->d_cl_out.as<int32_t>(), *ced = crow + std::max<int64_t>(nu, 1);
    const uint8_t *cstrand = (const uint8_t *)(ced + std::max<int64_t>(nu, 1));
    if (nu && centroid_row_of_unique) CUDA_TRY(c, cudaMemcpyAsync(centroid_row_of_unique, crow, (size_t)nu * 4, cudaMemcpyDefault, st));
    if (nu && strand_of_unique) CUDA_TRY(c, cudaMemcpyAsync(strand_of_unique, cstrand, (size_t)nu, cudaMemcpyDefault, st));
    if (nu && ed_of_unique) CUDA_TRY(c, cudaMemcpyAsync(ed_of_unique, ced, (size_t)nu * 4, cudaMemcpyDefault, st));
    if (nc && unique_of_row) CUDA_TRY(c, cudaMemcpyAsync(unique_of_row, c->d_cl_crow.p, (size_t)nc * 4, cudaMemcpyDefault, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return ITSX_OK;
}

int itsx_cluster_get_stats(const itsx_ctx *c, itsx_cluster_stats *st)
{
    CHECK_CTX(c);
    if (st) *st = c->clstats;
    return ITSX_OK;
}

int itsx_cluster_dtable(double id, int32_t lmax, int32_t *dmax)
{
    if (!(id > 0.5 && id <= 1.0) || lmax < 0 || !dmax) return ITSX_EINVAL;
    cluster_dtable(id, lmax, dmax);
    return ITSX_OK;
}

// ---- search ------------------------------------------------------------------------------------
void itsx_search_default_params(itsx_search_params *prm)
{
    prm->T = 10.0f;
    prm->F1 = prm->F2 = prm->F3 = 1e-6;
    prm->domE = 10.0;
    prm->resolve_multidomain = 1;
    prm->keep_rows = 0;
    prm->domz_upper = 0;
}
static int set_params(itsx_ctx *c, const itsx_search_params *prm)
{
    if (prm) c->prm = *prm;
    else itsx_search_default_params(&c->prm);
    if (!(c->prm.F1 >= 0 && c->prm.F2 >= 0 && c->prm.F3 >= 0)) { c->err = "search: negative filter threshold"; return ITSX_EINVAL; }
    return ITSX_OK;
}
int itsx_search_stage1(itsx_ctx *c, const itsx_search_params *prm)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    int rc = set_params(c, prm);
    if (rc) return rc;
    return search_stage1(c);
}
int itsx_search_seqs_stage1(itsx_ctx *c, const uint8_t *seq, const int64_t *off, int64_t nseq,
                            const itsx_search_params *prm)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    int rc = set_params(c, prm);
    if (rc) return rc;
    rc = search_build_seqs_from_host(c, seq, off, nseq);
    if (rc) return rc;
    return search_stage1(c);
}
int itsx_search_shard(itsx_ctx *c, int64_t first_unique, int64_t n_local)
{
    CHECK_CTX(c);
    c->shard_first = first_unique;
    c->shard_n = n_local;
    return ITSX_OK;
}
int itsx_nreported(itsx_ctx *c, int32_t *per_profile)
{
    CHECK_CTX(c);
    if (!c->stage1_done) { c->err = "nreported before search"; return ITSX_EINVAL; }
    if (per_profile) memcpy(per_profile, c->h_nrep.data(), c->h_nrep.size() * 4);     // [n_samples][P]
    return ITSX_OK;
}
int itsx_nreported_set(itsx_ctx *c, const int32_t *g)
{
    CHECK_CTX(c);
    if (!c->stage1_done) { c->err = "nreported_set before search stage1"; return ITSX_EINVAL; }
    c->h_nrep.assign(g, g + c->h_nrep.size());       // [n_samples][P] of the last stage 1
    return ITSX_OK;
}
int itsx_search_stage2(itsx_ctx *c)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    return search_stage2(c);
}
int itsx_search(itsx_ctx *c, const itsx_search_params *prm)
{
    int rc = itsx_search_stage1(c, prm);
    if (rc) return rc;
    return itsx_search_stage2(c);
}
int itsx_search_seqs(itsx_ctx *c, const uint8_t *seq, const int64_t *off, int64_t nseq, const itsx_search_params *prm)
{
    int rc = itsx_search_seqs_stage1(c, seq, off, nseq, prm);
    if (rc) return rc;
    return itsx_search_stage2(c);
}
int itsx_search_get_stats(const itsx_ctx *c, itsx_search_stats *st)
{
    CHECK_CTX(c);
    if (st) *st = c->sstats;
    return ITSX_OK;
}

int itsx_hits(itsx_ctx *c, itsx_dom_row *rows, int64_t cap, int64_t *n)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (!c->stage2_done) { c->err = "hits before search"; return ITSX_EINVAL; }
    // (compact mode, itsx_search_params.keep_rows: only the rows that were still undecided after stage 1 are here)
    std::vector<DomRec> h((size_t)c->ndom);
    if (c->ndom) {
        CUDA_TRY(c, cudaMemcpyAsync(h.data(), c->d_doms.p, (size_t)c->ndom * sizeof(DomRec), cudaMemcpyDefault, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    std::vector<int64_t> idx;
    idx.reserve(h.size());
    for (int64_t i = 0; i < (int64_t)h.size(); i++)
        if (h[i].pair_reported & 2) idx.push_back(i);
    // hmmsearch row order: profile; hit ln P ascending, then target index; domain position
    std::sort(idx.begin(), idx.end(), [&](int64_t a, int64_t b) {
        const DomRec &x = h[a], &y = h[b];
        if (x.prof != y.prof) return x.prof < y.prof;
        if (x.seq_lnP != y.seq_lnP) return x.seq_lnP < y.seq_lnP;
        if (x.seq != y.seq) return x.seq < y.seq;
        return x.dom_idx < y.dom_idx;
    });
    if (n) *n = (int64_t)idx.size();
    if (rows) {
        const int64_t m = std::min<int64_t>(cap, (int64_t)idx.size());
        for (int64_t i = 0; i < m; i++) {
            const DomRec &r = h[idx[i]];
            itsx_dom_row &o = rows[i];
            o.seq = r.seq; o.prof = r.prof; o.ienv = r.ienv; o.jenv = r.jenv; o.tlen = r.tlen; o.dom_idx = r.dom_idx;
            o.bitscore = r.bitscore; o.envsc = r.envsc; o.domcorrection = r.domcorrection; o.seq_score = r.seq_score;
            o.lnP = r.lnP; o.seq_lnP = r.seq_lnP; o.is_multidomain = r.is_multidomain; o.reported = 1;
        }
    }
    return ITSX_OK;
}

int itsx_positions(itsx_ctx *c, int32_t *start, int32_t *stop, int32_t *tlen,
                   int32_t *lsc, int32_t *lfrom, int32_t *lto, int32_t *rsc, int32_t *rfrom, int32_t *rto)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (!c->pos_valid) { c->err = "positions before search"; return ITSX_EINVAL; }
    int32_t *outs[9] = {start, stop, tlen, lsc, lfrom, lto, rsc, rfrom, rto};
    const int64_t n = c->npos;
    if (n == 0) return ITSX_OK;
    for (int k = 0; k < 9; k++)
        if (outs[k])
            CUDA_TRY(c, cudaMemcpyAsync(outs[k], c->d_pos.as<int32_t>() + (size_t)k * n, (size_t)n * 4, cudaMemcpyDefault, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    return ITSX_OK;
}

int itsx_positions_set(itsx_ctx *c, const int32_t *start, const int32_t *stop, const int32_t *tlen, int64_t n)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (n < 0 || (n && (!start || !stop || !tlen))) return ITSX_EINVAL;
    c->npos = n;
    CUDA_TRY(c, c->d_pos.ensure((size_t)std::max<int64_t>(n, 1) * 9 * 4));
    if (n) {
        CUDA_TRY(c, cudaMemsetAsync(c->d_pos.p, 0xff, (size_t)n * 9 * 4, c->stream));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_pos.as<int32_t>(), start, (size_t)n * 4, cudaMemcpyDefault, c->stream));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_pos.as<int32_t>() + n, stop, (size_t)n * 4, cudaMemcpyDefault, c->stream));
        CUDA_TRY(c, cudaMemcpyAsync(c->d_pos.as<int32_t>() + 2 * n, tlen, (size_t)n * 4, cudaMemcpyDefault, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    c->pos_valid = true;
    return ITSX_OK;
}

// ---- trim ------------------------------------------------------------------------------------------
int itsx_trim_set_map(itsx_ctx *c, const int32_t *uid, int64_t nreads, int64_t n_unique)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (nreads < 0 || n_unique < 0 || (nreads && !uid)) { c->err = "trim_set_map: bad argument"; return ITSX_EINVAL; }
    if (nreads >= 0x7fffffffLL) { c->err = "trim_set_map: more than 2^31-1 reads in one call"; return ITSX_ELIMIT; }
    CUDA_TRY(c, c->d_uid.ensure((size_t)std::max<int64_t>(nreads, 1) * 4));
    if (nreads) CUDA_TRY(c, cudaMemcpyAsync(c->d_uid.p, uid, (size_t)nreads * 4, cudaMemcpyDefault, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    c->nreads = nreads;
    c->n_unique = n_unique;
    c->cl_active = false;
    c->total_bases = 0;       // no resident read bytes: itsx_trim_* must be given seq/qual/off
    c->map_external = true;
    return ITSX_OK;
}

static int check_trim(itsx_ctx *c, int mode, int64_t nreads)
{
    if (c->stream_open) { c->err = "trim: a streamed upload is still open (itsx_reads_end)"; return ITSX_EINVAL; }
    if (mode < 0 || mode > 2) { c->err = "trim: mode must be 0, 1 or 2"; return ITSX_EINVAL; }
    if (nreads != c->nreads) { c->err = "trim: read count differs from the dereplicated set"; return ITSX_EINVAL; }
    if (c->npos != map_rows(c)) { c->err = "trim: position table does not cover every unique sequence"; return ITSX_EINVAL; }
    return ITSX_OK;
}

int itsx_trim_bounds(itsx_ctx *c, int mode, const int64_t *off_other, int64_t nreads,
                     uint8_t *keep, int32_t *lo, int32_t *hi, int64_t *n_kept)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    int rc = check_trim(c, mode, nreads);
    if (rc) return rc;
    if (c->map_external && !off_other) { c->err = "trim: offsets are required after itsx_trim_set_map"; return ITSX_EINVAL; }
    static thread_local DevBuf t_off, t_keep, t_lo, t_hi;
    CUDA_TRY(c, t_keep.ensure((size_t)nreads + 16));
    CUDA_TRY(c, t_lo.ensure((size_t)nreads * 4 + 16));
    CUDA_TRY(c, t_hi.ensure((size_t)nreads * 4 + 16));
    const int64_t *d_off = nullptr;
    if (off_other) {
        CUDA_TRY(c, t_off.ensure((size_t)(nreads + 1) * 8));
        CUDA_TRY(c, cudaMemcpyAsync(t_off.p, off_other, (size_t)(nreads + 1) * 8, cudaMemcpyDefault, c->stream));
        d_off = t_off.as<int64_t>();
    }
    rc = trim_bounds_dev(c, mode, d_off, nreads, t_keep.as<uint8_t>(), t_lo.as<int32_t>(), t_hi.as<int32_t>(), n_kept);
    if (rc) return rc;
    if (nreads) {
        if (keep) CUDA_TRY(c, cudaMemcpyAsync(keep, t_keep.p, (size_t)nreads, cudaMemcpyDefault, c->stream));
        if (lo) CUDA_TRY(c, cudaMemcpyAsync(lo, t_lo.p, (size_t)nreads * 4, cudaMemcpyDefault, c->stream));
        if (hi) CUDA_TRY(c, cudaMemcpyAsync(hi, t_hi.p, (size_t)nreads * 4, cudaMemcpyDefault, c->stream));
        CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    }
    return ITSX_OK;
}

int itsx_trim_gather(itsx_ctx *c, int mode, const uint8_t *seq, const uint8_t *qual, const int64_t *off,
                     int64_t nreads, int64_t *n_kept, int64_t *total,
                     int32_t *kept_index, int64_t *out_off, uint8_t *out_seq, uint8_t *out_qual)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    int rc = check_trim(c, mode, nreads);
    if (rc) return rc;
    if (!n_kept || !total) return ITSX_EINVAL;
    if (c->map_external && !off) { c->err = "trim: offsets are required after itsx_trim_set_map"; return ITSX_EINVAL; }
    if (c->map_external && !seq && (out_seq || out_off || kept_index)) {
        c->err = "trim: sequence bytes are required after itsx_trim_set_map";
        return ITSX_EINVAL;
    }
    static thread_local DevBuf t_off, t_seq, t_qual, t_keep, t_lo, t_hi, t_ki, t_oo, t_os, t_oq;
    cudaStream_t st = c->stream;
    const bool query = !out_seq && !out_off && !kept_index;
    CUDA_TRY(c, t_keep.ensure((size_t)nreads + 16));
    CUDA_TRY(c, t_lo.ensure((size_t)nreads * 4 + 16));
    CUDA_TRY(c, t_hi.ensure((size_t)nreads * 4 + 16));
    const int64_t *d_off = nullptr;
    const int64_t tot_in = (off && nreads) ? itsx_peek_i64(off + nreads) : 0;
    if (off) {
        CUDA_TRY(c, t_off.ensure((size_t)(nreads + 1) * 8));
        CUDA_TRY(c, cudaMemcpyAsync(t_off.p, off, (size_t)(nreads + 1) * 8, cudaMemcpyDefault, st));
        d_off = t_off.as<int64_t>();
    }
    int64_t nk = 0;
    rc = trim_bounds_dev(c, mode, d_off, nreads, t_keep.as<uint8_t>(), t_lo.as<int32_t>(), t_hi.as<int32_t>(), &nk);
    if (rc) return rc;
    if (query) {
        int64_t tot = 0;
        if (nreads) {
            CUDA_TRY(c, cudaMemcpyAsync(&tot, c->d_list2.as<int64_t>() + nreads, 8, cudaMemcpyDefault, st));
            CUDA_TRY(c, cudaStreamSynchronize(st));
        }
        *n_kept = nk;
        *total = tot;
        return ITSX_OK;
    }
    const uint8_t *d_seq = c->d_ascii.as<uint8_t>();
    const uint8_t *d_qual = nullptr;
    if (seq) {
        CUDA_TRY(c, t_seq.ensure((size_t)tot_in + 16));
        if (tot_in) CUDA_TRY(c, cudaMemcpyAsync(t_seq.p, seq, (size_t)tot_in, cudaMemcpyDefault, st));
        d_seq = t_seq.as<uint8_t>();
    }
    if (qual) {
        const int64_t tq = off ? tot_in : c->total_bases;
        CUDA_TRY(c, t_qual.ensure((size_t)tq + 16));
        if (tq) CUDA_TRY(c, cudaMemcpyAsync(t_qual.p, qual, (size_t)tq, cudaMemcpyDefault, st));
        d_qual = t_qual.as<uint8_t>();
    } else if (!seq && !off && c->qual_resident) {
        d_qual = c->d_qual.as<uint8_t>();       // qualities of the resident reads (itsx_quals_upload)
    }
    rc = trim_gather_dev(c, d_seq, d_qual, d_off ? d_off : c->d_off.as<int64_t>(), nreads, t_keep.as<uint8_t>(),
                         t_lo.as<int32_t>(), t_hi.as<int32_t>(), n_kept, total, t_ki, t_oo, t_os, t_oq);
    if (rc) return rc;
    if (kept_index && *n_kept) CUDA_TRY(c, cudaMemcpyAsync(kept_index, t_ki.p, (size_t)*n_kept * 4, cudaMemcpyDefault, st));
    if (out_off) CUDA_TRY(c, cudaMemcpyAsync(out_off, t_oo.p, (size_t)(*n_kept + 1) * 8, cudaMemcpyDefault, st));
    if (out_seq && *total) CUDA_TRY(c, cudaMemcpyAsync(out_seq, t_os.p, (size_t)*total, cudaMemcpyDefault, st));
    if (out_qual && d_qual && *total) CUDA_TRY(c, cudaMemcpyAsync(out_qual, t_oq.p, (size_t)*total, cudaMemcpyDefault, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return ITSX_OK;
}

int itsx_trim_gather_resident(itsx_ctx *c, int mode, int64_t *n_kept, int64_t *total)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    const int64_t n = c->nreads;
    int rc = check_trim(c, mode, n);
    if (rc) return rc;
    if (c->map_external) { c->err = "trim_gather_resident: no reads are resident"; return ITSX_EINVAL; }
    CUDA_TRY(c, c->r_keep.ensure((size_t)n + 16));
    CUDA_TRY(c, c->r_lo.ensure((size_t)n * 4 + 16));
    CUDA_TRY(c, c->r_hi.ensure((size_t)n * 4 + 16));
    int64_t nk = 0, nk2 = 0, tot = 0;
    rc = trim_bounds_dev(c, mode, nullptr, n, c->r_keep.as<uint8_t>(), c->r_lo.as<int32_t>(), c->r_hi.as<int32_t>(), &nk);
    if (rc) return rc;
    rc = trim_gather_dev(c, c->d_ascii.as<uint8_t>(), c->qual_resident ? c->d_qual.as<uint8_t>() : nullptr,
                         c->d_off.as<int64_t>(), n, c->r_keep.as<uint8_t>(), c->r_lo.as<int32_t>(), c->r_hi.as<int32_t>(),
                         &nk2, &tot, c->r_ki, c->r_oo, c->r_os, c->r_oq);
    if (rc) return rc;
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    c->r_nkept = nk2;
    c->r_total = tot;
    c->r_gathered = true;
    if (n_kept) *n_kept = nk2;
    if (total) *total = tot;
    return ITSX_OK;
}

// ---- whole path ------------------------------------------------------------------------------------------
// derep -> search -> positions -> trim bounds [-> re-expansion of the kept slices when the qualities are resident]
// events of a whole-path call: 0 start, 1 reads resident, 2 derep done, 3 search done, 4 trim done, 5 end, 6 gather done
typedef Timeline<7> RunTimeline;

static int run_device_part(itsx_ctx *c, const itsx_search_params *prm, itsx_run_stats *rs, const RunTimeline &tl)
{
    cudaStream_t st = c->stream;
    CUDA_TRY(c, tl.record(1, st));
    int rc = derep_run(c);
    if (rc) return rc;
    c->shard_first = 0;
    c->shard_n = -1;
    rc = search_build_seqs_from_derep(c);
    if (rc) return rc;
    CUDA_TRY(c, tl.record(2, st));
    rc = set_params(c, prm);
    if (rc) return rc;
    rc = search_stage1(c);
    if (rc) return rc;
    rc = search_stage2(c);
    if (rc) return rc;
    CUDA_TRY(c, tl.record(3, st));
    const int64_t n = c->nreads;
    CUDA_TRY(c, c->r_keep.ensure((size_t)n + 16));
    CUDA_TRY(c, c->r_lo.ensure((size_t)n * 4 + 16));
    CUDA_TRY(c, c->r_hi.ensure((size_t)n * 4 + 16));
    int64_t nk = 0;
    rc = trim_bounds_dev(c, 0, nullptr, n, c->r_keep.as<uint8_t>(), c->r_lo.as<int32_t>(), c->r_hi.as<int32_t>(), &nk);
    if (rc) return rc;
    CUDA_TRY(c, tl.record(4, st));
    rs->n_reads = n;
    rs->n_unique = c->n_unique;
    rs->n_kept = nk;
    c->r_nkept = nk;
    c->r_total = 0;
    c->r_gathered = false;
    if (n) {
        int64_t tot = 0;
        CUDA_TRY(c, cudaMemcpyAsync(&tot, c->d_list2.as<int64_t>() + n, 8, cudaMemcpyDefault, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        rs->out_bytes = tot;
        c->r_total = tot;
    }
    if (c->qual_resident) {
        int64_t nk2 = 0, tot2 = 0;
        rc = trim_gather_dev(c, c->d_ascii.as<uint8_t>(), c->d_qual.as<uint8_t>(), c->d_off.as<int64_t>(), n,
                             c->r_keep.as<uint8_t>(), c->r_lo.as<int32_t>(), c->r_hi.as<int32_t>(), &nk2, &tot2,
                             c->r_ki, c->r_oo, c->r_os, c->r_oq);
        if (rc) return rc;
        c->r_gathered = true;
    }
    CUDA_TRY(c, tl.record(6, st));
    return ITSX_OK;
}

static void run_times(itsx_run_stats &rs, const RunTimeline &tl, bool with_copies)
{
    if (with_copies) rs.ms_h2d = tl.ms(0, 1);
    rs.ms_derep = tl.ms(1, 2);
    rs.ms_search = tl.ms(2, 3);
    rs.ms_trim = tl.ms(3, 4);
    rs.ms_gather = tl.ms(4, 6);
    if (with_copies) rs.ms_d2h = tl.ms(6, 5);
    rs.ms_total = tl.ms(0, 5);
}

int itsx_quals_upload(itsx_ctx *c, const uint8_t *qual)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (c->map_external) { c->err = "quals_upload: no reads are resident (itsx_reads_upload first)"; return ITSX_EINVAL; }
    if (c->total_bases && !qual) { c->err = "quals_upload: null buffer"; return ITSX_EINVAL; }
    CUDA_TRY(c, c->d_qual.ensure((size_t)c->total_bases + 64));
    if (c->total_bases) CUDA_TRY(c, cudaMemcpyAsync(c->d_qual.p, qual, (size_t)c->total_bases, cudaMemcpyDefault, c->stream));
    CUDA_TRY(c, cudaStreamSynchronize(c->stream));
    c->qual_resident = true;
    return ITSX_OK;
}

int itsx_run(itsx_ctx *c, const uint8_t *seq, const int64_t *off, int64_t nreads, const itsx_search_params *prm,
             int32_t *rep_index, uint8_t *keep, int32_t *lo, int32_t *hi, itsx_run_stats *out)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    itsx_run_stats rs{};
    RunTimeline tl;
    CUDA_TRY(c, tl.status);
    cudaStream_t st = c->stream;
    CUDA_TRY(c, tl.record(0, st));
    int rc = itsx_reads_upload(c, seq, off, nreads);
    if (!rc) rc = run_device_part(c, prm, &rs, tl);
    if (!rc && nreads) {
        if (rep_index) CUDA_TRY(c, cudaMemcpyAsync(rep_index, c->d_rep.p, (size_t)nreads * 4, cudaMemcpyDefault, st));
        if (keep) CUDA_TRY(c, cudaMemcpyAsync(keep, c->r_keep.p, (size_t)nreads, cudaMemcpyDefault, st));
        if (lo) CUDA_TRY(c, cudaMemcpyAsync(lo, c->r_lo.p, (size_t)nreads * 4, cudaMemcpyDefault, st));
        if (hi) CUDA_TRY(c, cudaMemcpyAsync(hi, c->r_hi.p, (size_t)nreads * 4, cudaMemcpyDefault, st));
    }
    if (!rc) {
        CUDA_TRY(c, tl.record(5, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        run_times(rs, tl, true);
        if (out) *out = rs;
    }
    return rc;
}

int itsx_run_resident(itsx_ctx *c, const itsx_search_params *prm, itsx_run_stats *out)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    itsx_run_stats rs{};
    RunTimeline tl;
    CUDA_TRY(c, tl.status);
    cudaStream_t st = c->stream;
    CUDA_TRY(c, tl.record(0, st));
    int rc = run_device_part(c, prm, &rs, tl);
    if (!rc) {
        CUDA_TRY(c, tl.record(5, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        run_times(rs, tl, false);
        if (out) *out = rs;
    }
    return rc;
}

int itsx_run_fetch(itsx_ctx *c, int64_t *n_kept, int64_t *total, int32_t *kept_index, int64_t *out_off,
                   uint8_t *out_seq, uint8_t *out_qual)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (!c->r_gathered) { c->err = "run_fetch: no gathered output is resident (qualities were not uploaded)"; return ITSX_EINVAL; }
    cudaStream_t st = c->stream;
    const int64_t nk = c->r_nkept, tot = c->r_total;
    if (n_kept) *n_kept = nk;
    if (total) *total = tot;
    if (kept_index && nk) CUDA_TRY(c, cudaMemcpyAsync(kept_index, c->r_ki.p, (size_t)nk * 4, cudaMemcpyDefault, st));
    if (out_off) CUDA_TRY(c, cudaMemcpyAsync(out_off, c->r_oo.p, (size_t)(nk + 1) * 8, cudaMemcpyDefault, st));
    if (out_seq && tot) CUDA_TRY(c, cudaMemcpyAsync(out_seq, c->r_os.p, (size_t)tot, cudaMemcpyDefault, st));
    if (out_qual && tot && c->qual_resident) CUDA_TRY(c, cudaMemcpyAsync(out_qual, c->r_oq.p, (size_t)tot, cudaMemcpyDefault, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return ITSX_OK;
}

int itsx_run_trim(itsx_ctx *c, const uint8_t *seq, const uint8_t *qual, const int64_t *off, int64_t nreads,
                  const itsx_search_params *prm, int32_t *rep_index, int32_t *kept_index, int64_t *out_off,
                  uint8_t *out_seq, uint8_t *out_qual, itsx_run_stats *out)
{
    CHECK_CTX(c);
    CUDA_TRY(c, cudaSetDevice(c->device));
    if (nreads > 0 && !qual) { c->err = "run_trim: qualities are required"; return ITSX_EINVAL; }
    itsx_run_stats rs{};
    RunTimeline tl;
    CUDA_TRY(c, tl.status);
    cudaStream_t st = c->stream;
    CUDA_TRY(c, tl.record(0, st));
    int rc = itsx_reads_upload(c, seq, off, nreads);
    if (!rc) rc = itsx_quals_upload(c, qual);
    if (!rc) rc = run_device_part(c, prm, &rs, tl);
    if (!rc) {
        const int64_t nk = c->r_nkept, tot = c->r_total;
        if (rep_index && nreads) CUDA_TRY(c, cudaMemcpyAsync(rep_index, c->d_rep.p, (size_t)nreads * 4, cudaMemcpyDefault, st));
        if (kept_index && nk) CUDA_TRY(c, cudaMemcpyAsync(kept_index, c->r_ki.p, (size_t)nk * 4, cudaMemcpyDefault, st));
        if (out_off) CUDA_TRY(c, cudaMemcpyAsync(out_off, c->r_oo.p, (size_t)(nk + 1) * 8, cudaMemcpyDefault, st));
        if (out_seq && tot) CUDA_TRY(c, cudaMemcpyAsync(out_seq, c->r_os.p, (size_t)tot, cudaMemcpyDefault, st));
        if (out_qual && tot) CUDA_TRY(c, cudaMemcpyAsync(out_qual, c->r_oq.p, (size_t)tot, cudaMemcpyDefault, st));
        CUDA_TRY(c, tl.record(5, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        run_times(rs, tl, true);
        if (out) *out = rs;
    }
    return rc;
}

}  // extern "C"
