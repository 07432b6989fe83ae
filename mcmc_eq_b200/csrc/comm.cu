// comm.cu -- what spans more than one GPU: chain sharding, the posterior reduction and parallel-tempering swaps.
//
// Chains are independent (the reference runs them as separate processes, run/srun_mcmc_eq.sh:13,35), so the data path
// has no collective.  NCCL (over NVLink / NVSwitch) is used in exactly two places, both off the critical path:
//   * mq_posterior_allreduce: sum of the posterior accumulators (histograms of src/analyse_eq.c:589-606 and the
//     moment sums of :612-640) over all ranks, once at the end of a run -- two ncclAllReduce calls;
//   * mq_temper_swap: optional parallel tempering.  One ncclAllGather of (log-likelihood, beta) per chain (16 B x
//     chains), then every rank takes the same swap decisions from a shared counter-based random stream and swaps
//     TEMPERATURES, never states.  Not reference behaviour (the reference has no chain interaction); off by default.
// NCCL is bound at run time (dlopen of libnccl.so.2: the copy torch has already loaded when the host is Python, the
// system's otherwise), so the library loads on machines without it and single-GPU use never touches it.
#include <dlfcn.h>
#include <nccl.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../include/mcmceq_b200.h"
#include "errors.h"
#include "launch_count.h"
#include "state.h"

namespace mq {

struct Nccl {
    void* lib;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*);
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
    const char* (*GetErrorString)(ncclResult_t);
};

static Nccl* nccl()
{
    static Nccl N;
    static int state = 0;   // 0 untried, 1 ok, -1 failed
    if (state == 0) {
        state = -1;
        const char* names[] = {"libnccl.so.2", "libnccl.so", nullptr};
        for (int i = 0; names[i] && !N.lib; i++) N.lib = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
        if (N.lib) {
            N.GetUniqueId = (decltype(N.GetUniqueId))dlsym(N.lib, "ncclGetUniqueId");
            N.CommInitRank = (decltype(N.CommInitRank))dlsym(N.lib, "ncclCommInitRank");
            N.CommDestroy = (decltype(N.CommDestroy))dlsym(N.lib, "ncclCommDestroy");
            N.AllReduce = (decltype(N.AllReduce))dlsym(N.lib, "ncclAllReduce");
            N.AllGather = (decltype(N.AllGather))dlsym(N.lib, "ncclAllGather");
            N.GetErrorString = (decltype(N.GetErrorString))dlsym(N.lib, "ncclGetErrorString");
            if (N.GetUniqueId && N.CommInitRank && N.CommDestroy && N.AllReduce && N.AllGather && N.GetErrorString) state = 1;
        }
    }
    return state == 1 ? &N : nullptr;
}

struct Comm {
    ncclComm_t comm;
    int rank, world;
    double* gather;   // [world * n][2] (full log-likelihood, beta) of every chain of the job
};

#define MQ_NCCL(x)                                                                                   \
    do {                                                                                             \
        ncclResult_t r_ = (x);                                                                       \
        if (r_ != ncclSuccess) { set_error("%s: %s", #x, nccl()->GetErrorString(r_)); return MQ_ERR_CUDA; } \
    } while (0)

// ---- tempering kernels ------------------------------------------------------------------------------------
// full log-likelihood of the current state: -misfit/2 - sum_c n_c ln sigma_c (the sigma-dependent normalisation the
// noise arm accounts for through log_fac, src/mcmc_eq.c:1114-1117)
__global__ void temper_pack_kernel(int n, const double* ll, const float* noise, const float* beta, const int* n_class8,
                                   double* out)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    double L = ll[c];
    for (int k = 0; k < 8; k++) L -= (double)n_class8[k] * log((double)noise[8 * (size_t)c + k]);
    out[2 * (size_t)c] = L;
    out[2 * (size_t)c + 1] = beta ? (double)beta[c] : 1.0;
}

__device__ __forceinline__ uint32_t philox_word(uint64_t seed, uint32_t a, uint64_t b)
{   // one Philox4x32-10 block keyed by seed, counter (b, a, "swap")
    uint32_t c0 = (uint32_t)b, c1 = (uint32_t)(b >> 32), c2 = a, c3 = 0x73776170u, k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c0;
}

// Pairs (2k + parity, 2k + 1 + parity) of the global chain numbering, parity = round & 1.  Both members of a pair
// (possibly on different GPUs) evaluate the same test on the same gathered numbers with the same uniform deviate:
// swap iff log u < (beta_a - beta_b) (L_b - L_a).  A swap exchanges the temperatures.
__global__ void temper_swap_kernel(int n, long long first, long long total, uint64_t seed, long long round, const double* all,
                                   float* beta, int* n_swapped)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    const long long g = first + c, par = round & 1;
    if (g < par) return;
    const long long partner = ((g - par) ^ 1) + par;
    if (partner >= total) return;
    const long long lo = g < partner ? g : partner, hi = g < partner ? partner : g;
    const double La = all[2 * lo], Ba = all[2 * lo + 1], Lb = all[2 * hi], Bb = all[2 * hi + 1];
    const float u = ((float)(philox_word(seed, (uint32_t)lo, (uint64_t)round) >> 1) + 1.0f) / 2147483648.0f;   // (0, 1]
    if (Ba != Bb && log((double)u) < (Ba - Bb) * (Lb - La)) {   // equal temperatures: nothing to exchange
        beta[c] = (float)all[2 * partner + 1];
        if (g == lo) atomicAdd(n_swapped, 1);
    }
}

}  // namespace mq

using namespace mq;

extern "C" int mq_set_chain_offset(mq_handle* hh, int64_t first_chain)
{
    if (!hh || first_chain < 0) { set_error("mq_set_chain_offset: bad argument"); return MQ_ERR_ARG; }
    hh->h.chain_offset = first_chain;
    return MQ_OK;
}

static int ensure_beta(Handle* h)
{
    if (h->beta) return MQ_OK;
    MQ_CUDA(cudaMalloc((void**)&h->beta, h->n * sizeof(float)));
    std::vector<float> one(h->n, 1.0f);
    MQ_CUDA(cudaMemcpy(h->beta, one.data(), h->n * sizeof(float), cudaMemcpyHostToDevice));
    return MQ_OK;
}

extern "C" int mq_set_beta(mq_handle* hh, const float* beta)
{
    if (!hh || !beta) { set_error("mq_set_beta: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    for (int c = 0; c < h->n; c++)
        if (!(beta[c] > 0.f) || beta[c] > 1.f) { set_error("mq_set_beta: chain %d: beta %g outside (0, 1]", c, beta[c]); return MQ_ERR_ARG; }
    MQ_CUDA(cudaSetDevice(h->device));
    int rc = ensure_beta(h);
    if (rc != MQ_OK) return rc;
    MQ_CUDA(cudaMemcpyAsync(h->beta, beta, h->n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    MQ_CUDA(cudaStreamSynchronize(h->stream));
    return MQ_OK;
}

extern "C" int mq_get_beta(mq_handle* hh, float* beta)
{
    if (!hh || !beta) { set_error("mq_get_beta: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    MQ_CUDA(cudaSetDevice(h->device));
    if (!h->beta) { for (int c = 0; c < h->n; c++) beta[c] = 1.0f; return MQ_OK; }
    MQ_CUDA(cudaMemcpyAsync(beta, h->beta, h->n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    MQ_CUDA(cudaStreamSynchronize(h->stream));
    return MQ_OK;
}

// ---- posterior accumulators ---------------------------------------------------------------------------------
extern "C" int mq_posterior_begin(mq_handle* hh, float dv, float dvpvs, int64_t burn_in, mq_posterior_dims* dims)
{
    if (!hh || !(dv > 0.f) || !(dvpvs > 0.f)) { set_error("mq_posterior_begin: bad argument"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    MQ_CUDA(cudaSetDevice(h->device));
    Posterior& P = h->post;
    cudaFree(P.iblock); cudaFree(P.dblock);
    memset(&P, 0, sizeof P);
    P.dv = dv; P.dvpvs = dvpvs; P.burn_in = burn_in;
    P.ndv = (int)((h->cfg.vpmax - h->cfg.vpmin) / dv) + 1;            // src/analyse_eq.c:427-430
    P.ndvpvs = (int)((h->cfg.vpvsmax - h->cfg.vpvsmin) / dvpvs) + 1;
    P.n_int = (size_t)(P.ndv + P.ndvpvs + 1) * h->nz;
    P.n_dbl = 4 * (size_t)h->nz + 8 * (size_t)h->ne + 4 * (size_t)h->ns + 17;
    MQ_CUDA(cudaMalloc((void**)&P.iblock, P.n_int * sizeof(int32_t)));
    MQ_CUDA(cudaMalloc((void**)&P.dblock, P.n_dbl * sizeof(double)));
    MQ_CUDA(cudaMemsetAsync(P.iblock, 0, P.n_int * sizeof(int32_t), h->stream));
    MQ_CUDA(cudaMemsetAsync(P.dblock, 0, P.n_dbl * sizeof(double), h->stream));
    MQ_CUDA(cudaStreamSynchronize(h->stream));
    P.on = 1;
    if (dims) { dims->ndv = P.ndv; dims->ndvpvs = P.ndvpvs; dims->nz = h->nz; dims->n_events = h->ne; dims->n_stations = h->ns; }
    return MQ_OK;
}

extern "C" int mq_posterior_get(mq_handle* hh, int32_t* hist_vp, int32_t* hist_vpvs, int32_t* boundary, double* vsum,
                                double* eqsum, double* ressum, double* noisesum, int64_t* n_models)
{
    if (!hh) { set_error("mq_posterior_get: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    const Posterior& P = h->post;
    if (!P.on) { set_error("mq_posterior_get: mq_posterior_begin was not called"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const size_t nz = h->nz;
    const int32_t* ib = P.iblock;
    const double* db = P.dblock;
#define GET(dst, src, cnt) if (dst) MQ_CUDA(cudaMemcpyAsync(dst, src, (cnt) * sizeof(*(dst)), cudaMemcpyDeviceToHost, s))
    GET(hist_vp, ib, P.ndv * nz); GET(hist_vpvs, ib + P.ndv * nz, P.ndvpvs * nz); GET(boundary, ib + (P.ndv + P.ndvpvs) * nz, nz);
    GET(vsum, db, 4 * nz); GET(eqsum, db + 4 * nz, 8 * (size_t)h->ne); GET(ressum, db + 4 * nz + 8 * (size_t)h->ne, 4 * (size_t)h->ns);
    GET(noisesum, db + 4 * nz + 8 * (size_t)h->ne + 4 * (size_t)h->ns, 16);
#undef GET
    double cnt = 0;
    MQ_CUDA(cudaMemcpyAsync(&cnt, db + P.n_dbl - 1, sizeof(double), cudaMemcpyDeviceToHost, s));
    MQ_CUDA(cudaStreamSynchronize(s));
    if (n_models) *n_models = (int64_t)(cnt + 0.5);
    return MQ_OK;
}

// ---- NCCL communicator -------------------------------------------------------------------------------------------
extern "C" int mq_comm_unique_id(uint8_t* id)
{
    if (!id) { set_error("mq_comm_unique_id: null"); return MQ_ERR_ARG; }
    if (!nccl()) { set_error("mq_comm_unique_id: libnccl.so.2 not found"); return MQ_ERR_UNSUPPORTED; }
    ncclUniqueId u;
    MQ_NCCL(nccl()->GetUniqueId(&u));
    static_assert(sizeof(ncclUniqueId) == MQ_COMM_ID_BYTES, "ncclUniqueId size");
    memcpy(id, &u, sizeof u);
    return MQ_OK;
}

extern "C" int mq_comm_init(mq_handle* hh, const uint8_t* id, int rank, int world)
{
    if (!hh || !id || world < 1 || rank < 0 || rank >= world) { set_error("mq_comm_init: bad argument"); return MQ_ERR_ARG; }
    if (!nccl()) { set_error("mq_comm_init: libnccl.so.2 not found"); return MQ_ERR_UNSUPPORTED; }
    Handle* h = &hh->h;
    if (h->comm) { set_error("mq_comm_init: already initialised"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    ncclUniqueId u;
    memcpy(&u, id, sizeof u);
    Comm* c = new Comm();
    c->rank = rank; c->world = world; c->gather = nullptr; c->comm = nullptr;
    ncclResult_t r = nccl()->CommInitRank(&c->comm, world, u, rank);
    if (r != ncclSuccess) { set_error("ncclCommInitRank: %s", nccl()->GetErrorString(r)); delete c; return MQ_ERR_CUDA; }
    h->comm = c;
    h->chain_offset = (long long)rank * h->n;   // contiguous shards of equal size
    return MQ_OK;
}

extern "C" int mq_comm_destroy(mq_handle* hh)
{
    if (!hh) return MQ_OK;
    Handle* h = &hh->h;
    Comm* c = (Comm*)h->comm;
    if (!c) return MQ_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    if (c->comm && nccl()) nccl()->CommDestroy(c->comm);
    cudaFree(c->gather);
    delete c;
    h->comm = nullptr;
    return MQ_OK;
}

extern "C" int mq_posterior_allreduce(mq_handle* hh)
{
    if (!hh) { set_error("mq_posterior_allreduce: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    Comm* c = (Comm*)h->comm;
    if (!h->post.on) { set_error("mq_posterior_allreduce: mq_posterior_begin was not called"); return MQ_ERR_STATE; }
    if (!c) { set_error("mq_posterior_allreduce: mq_comm_init was not called"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    MQ_NCCL(nccl()->AllReduce(h->post.iblock, h->post.iblock, h->post.n_int, ncclInt32, ncclSum, c->comm, h->stream));
    MQ_NCCL(nccl()->AllReduce(h->post.dblock, h->post.dblock, h->post.n_dbl, ncclFloat64, ncclSum, c->comm, h->stream));
    MQ_CUDA(cudaStreamSynchronize(h->stream));
    return MQ_OK;
}

extern "C" int mq_temper_swap(mq_handle* hh, int64_t round, int32_t* n_swapped)
{
    if (!hh || round < 0) { set_error("mq_temper_swap: bad argument"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    if (!h->forward_done) { set_error("mq_temper_swap: no likelihood yet (mq_init_chains / mq_forward first)"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    int rc = ensure_beta(h);
    if (rc != MQ_OK) return rc;
    Comm* c = (Comm*)h->comm;
    const int world = c ? c->world : 1, rank = c ? c->rank : 0;
    const size_t n = h->n, total = n * world;
    double* all = nullptr;
    static_assert(sizeof(int) == sizeof(int32_t), "int");
    int* d_scr = nullptr;    // [8 class counts | swap counter]
    MQ_CUDA(cudaMalloc((void**)&d_scr, 9 * sizeof(int)));
    int scr[9];
    for (int k = 0; k < 8; k++) scr[k] = h->n_class[k];
    scr[8] = 0;
    MQ_CUDA(cudaMemcpyAsync(d_scr, scr, sizeof scr, cudaMemcpyHostToDevice, h->stream));
    if (c) {
        if (!c->gather) MQ_CUDA(cudaMalloc((void**)&c->gather, total * 2 * sizeof(double)));
        all = c->gather;
    } else {
        MQ_CUDA(cudaMalloc((void**)&all, total * 2 * sizeof(double)));
    }
    double* mine = all + 2 * n * rank;
    temper_pack_kernel<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>((int)n, h->ll, h->noise, h->beta, d_scr, mine);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    if (c && world > 1) MQ_NCCL(nccl()->AllGather(mine, all, 2 * n, ncclFloat64, c->comm, h->stream));
    temper_swap_kernel<<<(unsigned)((n + 127) / 128), 128, 0, h->stream>>>((int)n, (long long)(n * rank), (long long)total, h->seed,
                                                                           (long long)round, all, h->beta, d_scr + 8);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    MQ_CUDA(cudaMemcpyAsync(scr, d_scr, sizeof scr, cudaMemcpyDeviceToHost, h->stream));
    MQ_CUDA(cudaStreamSynchronize(h->stream));
    if (n_swapped) *n_swapped = scr[8];
    cudaFree(d_scr);
    if (!c) cudaFree(all);
    return MQ_OK;
}

namespace mq {
int comm_allreduce_sum(Handle* h, double* buf, size_t count)
{
    Comm* c = (Comm*)h->comm;
    if (!c || c->world < 2) return MQ_OK;
    MQ_NCCL(nccl()->AllReduce(buf, buf, count, ncclFloat64, ncclSum, c->comm, h->stream));
    return MQ_OK;
}

void comm_destroy(Handle* h)
{
    mq_handle* hh = reinterpret_cast<mq_handle*>(h);   // Handle is the first and only member of mq_handle
    mq_comm_destroy(hh);
    cudaFree(h->beta); h->beta = nullptr;
    cudaFree(h->post.iblock); cudaFree(h->post.dblock);
    memset(&h->post, 0, sizeof h->post);
}
}  // namespace mq
