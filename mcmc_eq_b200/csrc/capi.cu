// capi.cu -- C ABI: handle life cycle, model upload/download, batched forward (mq_forward).
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../include/mcmceq_b200.h"
#include "chain.cuh"
#include "eikonal.cuh"
#include "errors.h"
#include "forward.cuh"
#include "launch_count.h"
#include "state.h"

using namespace mq;

namespace {

template <class T>
cudaError_t dalloc(T** p, size_t count)
{
    cudaError_t e = cudaMalloc((void**)p, (count ? count : 1) * sizeof(T));
    if (e == cudaSuccess) e = cudaMemset(*p, 0, (count ? count : 1) * sizeof(T));
    return e;
}
template <class T>
cudaError_t h2d(T* dst, const T* src, size_t count, cudaStream_t s)
{
    return cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyHostToDevice, s);
}
template <class T>
cudaError_t d2h(T* dst, const T* src, size_t count, cudaStream_t s)
{
    return cudaMemcpyAsync(dst, src, count * sizeof(T), cudaMemcpyDeviceToHost, s);
}

cudaError_t alloc_view(EvalView* v, int n)
{
    cudaError_t e;
    if ((e = dalloc(&v->mbuf, n))) return e;
    if ((e = dalloc(&v->tbuf, 2 * (size_t)n))) return e;
    if ((e = dalloc(&v->ebuf, n))) return e;
    if ((e = dalloc(&v->q_idx, n))) return e;
    if ((e = dalloc(&v->q_xyz, 3 * (size_t)n))) return e;
    if ((e = dalloc(&v->r_idx, n))) return e;
    if ((e = dalloc(&v->r_d, 4 * (size_t)n))) return e;
    if ((e = dalloc(&v->ev_only, n))) return e;
    v->pres_over = nullptr; v->sres_over = nullptr; v->hold = nullptr;
    return cudaSuccess;
}
void free_view(EvalView* v)
{
    cudaFree(v->mbuf); cudaFree(v->tbuf); cudaFree(v->ebuf); cudaFree(v->q_idx);
    cudaFree(v->q_xyz); cudaFree(v->r_idx); cudaFree(v->r_d); cudaFree(v->ev_only);
}

// current-state view: evaluate what is stored, write where it is stored
__global__ void sync_cur_view(int n, const int32_t* mcur, const int32_t* tcur, const int32_t* ecur, EvalView v)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    v.mbuf[c] = mcur[c];
    v.tbuf[2 * c] = tcur[2 * c];
    v.tbuf[2 * c + 1] = tcur[2 * c + 1];
    v.ebuf[c] = ecur[c];
    v.q_idx[c] = -1;
    v.r_idx[c] = -1;
    v.ev_only[c] = -1;
}

// mf <- mf_eval and likelihood of the current models (src/mcmc_eq.c:749-756)
__global__ void adopt_totals_kernel(int n, int sum_of_picks, const float* mf_eval, const float* noise, float* mf,
                                    double* misfit, double* rms, double* ll)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    float m[8];
    for (int k = 0; k < 8; k++) { m[k] = mf_eval[8 * (size_t)c + k]; mf[8 * (size_t)c + k] = m[k]; }
    const float* s = noise + 8 * (size_t)c;
    misfit[c] = chain_misfit(m, s);
    rms[c] = chain_rms(m, sum_of_picks);
    ll[c] = -misfit[c] / 2.0;
}

}  // namespace

extern "C" int mq_destroy(mq_handle* hh)
{
    if (!hh) return MQ_OK;
    Handle* h = &hh->h;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    comm_destroy(h);
    diag_destroy(h);
    hypo_destroy(h);
    sampler_destroy(h);
    profile_destroy(h);
    cudaFree(h->pk.ev_off); cudaFree(h->pk.n_p); cudaFree(h->pk.st_id); cudaFree(h->pk.r0); cudaFree(h->pk.cp);
    cudaFree(h->pk.x); cudaFree(h->pk.y); cudaFree(h->pk.t); cudaFree(h->pk.w1); cudaFree(h->pk.w2); cudaFree(h->pk.fix);
    cudaFree(h->pk.rec4); cudaFree(h->pk.rec2);
    cudaFree(h->d_rows); cudaFree(h->d_all_rows);
    free(h->rows_host);
    cudaFree(h->dim); cudaFree(h->mcur); cudaFree(h->tcur); cudaFree(h->ecur);
    cudaFree(h->z); cudaFree(h->vp); cudaFree(h->vpvs); cudaFree(h->eq); cudaFree(h->pres); cudaFree(h->sres);
    cudaFree(h->noise); cudaFree(h->tab); cudaFree(h->evsum); cudaFree(h->origin); cudaFree(h->mf);
    cudaFree(h->ll); cudaFree(h->rms); cudaFree(h->misfit); cudaFree(h->err);
    free_view(&h->cur_view); free_view(&h->prop_view);
    cudaFree(h->evq); cudaFree(h->oq); cudaFree(h->mf_eval); cudaFree(h->resid); cudaFree(h->tpred);
    cudaFree(h->item_chain); cudaFree(h->item_phase); cudaFree(h->n_items); cudaFree(h->slow); cudaFree(h->item_tab);
    cudaFree(h->solve_status);
    eik_work_free(&h->eik);
    if (h->host_flags) cudaFreeHost(h->host_flags);
    if (h->flags_ev) cudaEventDestroy(h->flags_ev);
    for (int i = 0; i < 2; i++)
        for (int k = 0; k < 16; k++)
            if (h->timer_ev[i][k]) cudaEventDestroy(h->timer_ev[i][k]);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete hh;
    return MQ_OK;
}

extern "C" int mq_create(const mq_config* cfg, const mq_picks* pk, int n_chains, int device, uint64_t seed,
                         mq_handle** out)
{
    if (!cfg || !pk || !out || n_chains < 1) { set_error("mq_create: bad argument"); return MQ_ERR_ARG; }
    const mq_grid& g = cfg->grid;
    if (g.nz < 2 || g.nx < 1 || g.ny < 1 || !(g.h > 0.f)) { set_error("mq_create: bad grid"); return MQ_ERR_ARG; }
    if (cfg->tria != 0 && cfg->tria != 1) { set_error("mq_create: config line 29 (TRIA) must be 0 or 1"); return MQ_ERR_ARG; }
    if (pk->n_events < 1 || pk->n_picks < 1 || pk->n_stations < 1) { set_error("mq_create: empty pick set"); return MQ_ERR_ARG; }
    if (cfg->max_dim < 1) { set_error("mq_create: max_dim < 1"); return MQ_ERR_ARG; }
    *out = nullptr;
    MQ_CUDA(cudaSetDevice(device));

    mq_handle* hh = new mq_handle();
    Handle* h = &hh->h;
    memset(h, 0, sizeof *h);
    h->cfg = *cfg;
    h->device = device;
    h->seed = seed;
    h->picks_sum = picks_checksum(pk);
    h->n = n_chains;
    h->md = std::min(cfg->max_dim, 1000);   // MD, src/mc.h:49
    h->ne = pk->n_events; h->ns = pk->n_stations; h->np = pk->n_picks;
    h->nz = g.nz;
    h->nxmod = (int)sqrt((double)(g.nx * g.nx + g.ny * g.ny));   // src/mcmc_eq.c:520
    h->xp = (h->nxmod + 3) / 4 * 4;
    h->lvz_flag = cfg->inv_control > 0 ? 1 : 0;                  // src/mcmc_eq.c:374
    h->inv_control = cfg->inv_control > 0 ? -cfg->inv_control : cfg->inv_control;
    h->xmin = g.x0; h->xmax = g.x0 + (g.nx - 1) * g.h;           // src/mcmc_eq.c:397-402
    h->ymin = g.y0; h->ymax = g.y0 + (g.ny - 1) * g.h;
    h->zmin = g.z0; h->zmax = g.z0 + (g.nz - 1) * g.h;
    if (h->nxmod < 2) { set_error("mq_create: nxmod < 2"); delete hh; return MQ_ERR_ARG; }

    // ---- picks: receiver layer and elevation weights (src/mcmc_eq.c:503-517), class counts
    const int np = pk->n_picks, ne = pk->n_events;
    std::vector<int32_t> layer(np), cp(np), r0(np);
    std::vector<float> w1(np), w2(np);
    std::vector<char> keep(g.nz, 0);
    int max_ev = 0;
    for (int e = 0; e < ne; e++) {
        const int b = pk->ev_off[e], end = pk->ev_off[e + 1];
        if (end < b || end > np || pk->n_p[e] < 0 || pk->n_p[e] > end - b) { set_error("mq_create: bad ev_off/n_p at event %d", e); delete hh; return MQ_ERR_ARG; }
        if (end - b == 0) { set_error("mq_create: event %d has no picks", e); delete hh; return MQ_ERR_ARG; }
        max_ev = std::max(max_ev, end - b);
        for (int j = b; j < end; j++) {
            const int isS = (j - b) >= pk->n_p[e];
            const int cl = pk->cls[j];
            if (cl < 0 || cl > 3) { set_error("mq_create: pick class %d", cl); delete hh; return MQ_ERR_ARG; }
            if (pk->st_id[j] < 0 || pk->st_id[j] >= pk->n_stations) { set_error("mq_create: station id %d", pk->st_id[j]); delete hh; return MQ_ERR_ARG; }
            cp[j] = 2 * cl + isS;
            h->n_class[cp[j]]++;
            const float zs = pk->z[j];
            layer[j] = (int)((zs - g.z0) / g.h);
            w2[j] = -(layer[j] * g.h + g.z0 - zs) / g.h;
            w1[j] = 1.0 - w2[j];
            // the reference indexes ttt[layer] and ttt[layer+1] unchecked (src/misfit.c:91)
            if (layer[j] < 0 || layer[j] + 1 > g.nz - 1) { set_error("mq_create: station elevation %g outside the depth grid", zs); delete hh; return MQ_ERR_ARG; }
            keep[layer[j]] = keep[layer[j] + 1] = 1;
        }
    }
    h->sum_of_picks = np;
    std::vector<int32_t> rowidx(g.nz, -1);
    h->n_rows = 0;
    h->rows_host = (int32_t*)malloc(sizeof(int32_t) * g.nz);
    for (int j = 0; j < g.nz; j++)
        if (keep[j]) { rowidx[j] = h->n_rows; h->rows_host[h->n_rows++] = j; }
    for (int j = 0; j < np; j++) r0[j] = rowidx[layer[j]];
    h->tab_stride = (size_t)h->n_rows * h->nz * h->xp;

#define TRY(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { set_error("%s: %s", #x, cudaGetErrorString(e_)); mq_destroy(hh); return e_ == cudaErrorMemoryAllocation ? MQ_ERR_NOMEM : MQ_ERR_CUDA; } } while (0)
    TRY(cudaStreamCreate(&h->stream));
    cudaStream_t s = h->stream;
    const size_t n = n_chains;
    h->pk.n_events = ne; h->pk.n_picks = np; h->pk.max_event_picks = max_ev;
    TRY(dalloc(&h->pk.ev_off, ne + 1)); TRY(h2d(h->pk.ev_off, pk->ev_off, ne + 1, s));
    TRY(dalloc(&h->pk.n_p, ne));        TRY(h2d(h->pk.n_p, pk->n_p, ne, s));
    TRY(dalloc(&h->pk.st_id, np));      TRY(h2d(h->pk.st_id, pk->st_id, np, s));
    TRY(dalloc(&h->pk.r0, np));         TRY(h2d(h->pk.r0, r0.data(), np, s));
    TRY(dalloc(&h->pk.cp, np));         TRY(h2d(h->pk.cp, cp.data(), np, s));
    TRY(dalloc(&h->pk.x, np));          TRY(h2d(h->pk.x, pk->x, np, s));
    TRY(dalloc(&h->pk.y, np));          TRY(h2d(h->pk.y, pk->y, np, s));
    TRY(dalloc(&h->pk.t, np));          TRY(h2d(h->pk.t, pk->t, np, s));
    TRY(dalloc(&h->pk.w1, np));         TRY(h2d(h->pk.w1, w1.data(), np, s));
    TRY(dalloc(&h->pk.w2, np));         TRY(h2d(h->pk.w2, w2.data(), np, s));
    {
        std::vector<float4> rec4(np);
        std::vector<float2> rec2(np);
        for (int j = 0; j < np; j++) {
            if (pk->st_id[j] < 0 || pk->st_id[j] >= (1 << 20) || r0[j] < 0 || r0[j] >= 256 || cp[j] < 0 || cp[j] >= 8) {
                set_error("mq_create: pick %d does not fit the packed record (station %d, row %d, class %d)", j, pk->st_id[j], r0[j], cp[j]);
                mq_destroy(hh);
                return MQ_ERR_ARG;
            }
            const uint32_t code = (uint32_t)pk->st_id[j] | ((uint32_t)r0[j] << 20) | ((uint32_t)cp[j] << 28);
            float cf;
            memcpy(&cf, &code, sizeof cf);
            rec4[j] = make_float4(pk->x[j], pk->y[j], pk->t[j], (float)w1[j]);
            rec2[j] = make_float2((float)w2[j], cf);
        }
        TRY(dalloc(&h->pk.rec4, np));   TRY(h2d(h->pk.rec4, rec4.data(), np, s));
        TRY(dalloc(&h->pk.rec2, np));   TRY(h2d(h->pk.rec2, rec2.data(), np, s));
        TRY(cudaStreamSynchronize(s));
    }
    TRY(dalloc(&h->pk.fix, 3 * (size_t)ne));
    {
        std::vector<double> fix(3 * (size_t)ne, -9999.0);
        if (pk->fix) std::copy(pk->fix, pk->fix + 3 * (size_t)ne, fix.begin());
        TRY(h2d(h->pk.fix, fix.data(), fix.size(), s));
        TRY(cudaStreamSynchronize(s));
    }
    TRY(dalloc(&h->d_rows, h->n_rows)); TRY(h2d(h->d_rows, h->rows_host, h->n_rows, s));
    {
        std::vector<int32_t> all(g.nz);
        for (int j = 0; j < g.nz; j++) all[j] = j;
        TRY(dalloc(&h->d_all_rows, g.nz)); TRY(h2d(h->d_all_rows, all.data(), g.nz, s));
        TRY(cudaStreamSynchronize(s));
    }

    TRY(dalloc(&h->dim, 2 * n)); TRY(dalloc(&h->mcur, n)); TRY(dalloc(&h->tcur, 2 * n)); TRY(dalloc(&h->ecur, n));
    TRY(dalloc(&h->z, 2 * n * h->md)); TRY(dalloc(&h->vp, 2 * n * h->md)); TRY(dalloc(&h->vpvs, 2 * n * h->md));
    TRY(dalloc(&h->eq, n * ne * 3)); TRY(dalloc(&h->pres, n * h->ns)); TRY(dalloc(&h->sres, n * h->ns));
    TRY(dalloc(&h->noise, n * 8));
    TRY(dalloc(&h->tab, 2 * n * 2 * h->tab_stride));
    TRY(dalloc(&h->evsum, 2 * n * ne * 8)); TRY(dalloc(&h->origin, 2 * n * ne));
    TRY(dalloc(&h->mf, n * 8)); TRY(dalloc(&h->ll, n)); TRY(dalloc(&h->rms, n)); TRY(dalloc(&h->misfit, n));
    TRY(dalloc(&h->err, 1));
    TRY(cudaHostAlloc((void**)&h->host_flags, 2 * sizeof(int32_t), cudaHostAllocDefault));
    h->host_flags[0] = h->host_flags[1] = 0;
    TRY(cudaEventCreateWithFlags(&h->flags_ev, cudaEventDisableTiming));
    TRY(alloc_view(&h->cur_view, n_chains)); TRY(alloc_view(&h->prop_view, n_chains));
    TRY(dalloc(&h->evq, n * 8)); TRY(dalloc(&h->oq, n)); TRY(dalloc(&h->mf_eval, n * 8));
    // h->resid ([n][np] per-pick scratch) is allocated by launch_misfit when it is first needed
    TRY(dalloc(&h->item_chain, 2 * n)); TRY(dalloc(&h->item_phase, 2 * n)); TRY(dalloc(&h->n_items, 1));
    TRY(dalloc(&h->slow, 2 * n * h->nz)); TRY(dalloc(&h->item_tab, 2 * n)); TRY(dalloc(&h->solve_status, 1));
    TRY(eik_work_alloc(&h->eik, h->nxmod, h->nz, 2 * n_chains * h->nz, true, device));
    TRY(cudaStreamSynchronize(s));
#undef TRY
    *out = hh;
    return MQ_OK;
}

// sync: wait for the copies before returning (the caller may reuse its buffers at once); mq_forward_host goes on enqueueing
// the forward on the same stream and waits once, for the results
static int set_models(mq_handle* hh, const mq_models* m, bool sync)
{
    if (!hh || !m) { set_error("mq_set_models: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    if (m->n_chains != h->n || m->n_events != h->ne || m->n_stations != h->ns || m->max_dim > h->md || m->max_dim < 1) {
        set_error("mq_set_models: shape mismatch (chains %d/%d events %d/%d stations %d/%d max_dim %d/%d)", m->n_chains, h->n,
                  m->n_events, h->ne, m->n_stations, h->ns, m->max_dim, h->md);
        return MQ_ERR_ARG;
    }
    for (int c = 0; c < h->n; c++)
        if (m->dim[c] < 1 || m->dim[c] > m->max_dim) { set_error("mq_set_models: chain %d has dimension %d", c, m->dim[c]); return MQ_ERR_ARG; }
    MQ_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const size_t n = h->n;
    // models go into buffer 0; all buffer indices reset
    MQ_CUDA(cudaMemsetAsync(h->mcur, 0, n * sizeof(int32_t), s));
    MQ_CUDA(cudaMemsetAsync(h->tcur, 0, 2 * n * sizeof(int32_t), s));
    MQ_CUDA(cudaMemsetAsync(h->ecur, 0, n * sizeof(int32_t), s));
    MQ_CUDA(h2d(h->dim, m->dim, n, s));
    MQ_CUDA(cudaMemcpy2DAsync(h->z, h->md * sizeof(float), m->z, m->max_dim * sizeof(float), m->max_dim * sizeof(float), n, cudaMemcpyHostToDevice, s));
    MQ_CUDA(cudaMemcpy2DAsync(h->vp, h->md * sizeof(float), m->vp, m->max_dim * sizeof(float), m->max_dim * sizeof(float), n, cudaMemcpyHostToDevice, s));
    MQ_CUDA(cudaMemcpy2DAsync(h->vpvs, h->md * sizeof(float), m->vpvs, m->max_dim * sizeof(float), m->max_dim * sizeof(float), n, cudaMemcpyHostToDevice, s));
    MQ_CUDA(h2d(h->eq, m->eq, n * h->ne * 3, s));
    MQ_CUDA(h2d(h->pres, m->pres, n * h->ns, s));
    MQ_CUDA(h2d(h->sres, m->sres, n * h->ns, s));
    MQ_CUDA(h2d(h->noise, m->noise, n * 8, s));
    if (sync) MQ_CUDA(cudaStreamSynchronize(s));
    h->models_set = true;
    h->forward_done = false;
    return MQ_OK;
}
extern "C" int mq_set_models(mq_handle* hh, const mq_models* m) { return set_models(hh, m, true); }

extern "C" int mq_get_models(mq_handle* hh, mq_models* m)
{
    if (!hh || !m) { set_error("mq_get_models: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    if (m->n_chains != h->n || m->n_events != h->ne || m->n_stations != h->ns || m->max_dim < 1) {
        set_error("mq_get_models: shape mismatch"); return MQ_ERR_ARG;
    }
    MQ_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const size_t n = h->n;
    std::vector<int32_t> mcur(n), ecur(n), dim2(2 * n);
    MQ_CUDA(d2h(mcur.data(), h->mcur, n, s));
    MQ_CUDA(d2h(ecur.data(), h->ecur, n, s));
    MQ_CUDA(d2h(dim2.data(), h->dim, 2 * n, s));
    MQ_CUDA(cudaStreamSynchronize(s));
    const int w = std::min(m->max_dim, h->md);
    // both buffers of the double-buffered arrays in one copy each, the current one of every chain picked on the host
    // (four transfers whatever the number of chains)
    std::vector<float> z2(2 * n * h->md), vp2(2 * n * h->md), vpvs2(2 * n * h->md), org2;
    MQ_CUDA(d2h(z2.data(), h->z, z2.size(), s));
    MQ_CUDA(d2h(vp2.data(), h->vp, vp2.size(), s));
    MQ_CUDA(d2h(vpvs2.data(), h->vpvs, vpvs2.size(), s));
    if (m->origin) { org2.resize(2 * n * h->ne); MQ_CUDA(d2h(org2.data(), h->origin, org2.size(), s)); }
    MQ_CUDA(cudaStreamSynchronize(s));
    for (size_t c = 0; c < n; c++) {
        const size_t mo = ((size_t)mcur[c] * n + c) * h->md;
        m->dim[c] = dim2[mcur[c] * n + c];
        if (m->dim[c] > m->max_dim) { set_error("mq_get_models: chain %zu has %d nuclei > max_dim %d", c, m->dim[c], m->max_dim); return MQ_ERR_ARG; }
        memcpy(m->z + c * m->max_dim, z2.data() + mo, w * sizeof(float));
        memcpy(m->vp + c * m->max_dim, vp2.data() + mo, w * sizeof(float));
        memcpy(m->vpvs + c * m->max_dim, vpvs2.data() + mo, w * sizeof(float));
        if (m->origin) memcpy(m->origin + c * h->ne, org2.data() + ((size_t)ecur[c] * n + c) * h->ne, h->ne * sizeof(float));
    }
    MQ_CUDA(d2h(m->eq, h->eq, n * h->ne * 3, s));
    MQ_CUDA(d2h(m->pres, h->pres, n * h->ns, s));
    MQ_CUDA(d2h(m->sres, h->sres, n * h->ns, s));
    MQ_CUDA(d2h(m->noise, h->noise, n * 8, s));
    MQ_CUDA(cudaStreamSynchronize(s));
    return MQ_OK;
}

// ---- device error words -------------------------------------------------------------------------------------
// Kernels raise errors by setting bits of h->err (kErrStatcor, kErrRetry) or a negative h->solve_status.  Calls that
// return results to the host read them synchronously (check_device_errors); mq_step in lock-step mode stays asynchronous:
// it leaves a copy of the two words in pinned memory (flags_enqueue) and the next call that synchronises -- mq_sync,
// mq_get_stats, mq_drain, ... -- or the next mq_step that finds the copy complete reports them (flags_poll).
namespace mq {
static int decode_flags(Handle* h, int32_t err, int32_t status)
{
    if (err != 0) {
        cudaMemsetAsync(h->err, 0, sizeof(int32_t), h->stream);
        if (err & kErrStatcor) { set_error("ERROR points to invalid station correction (src/misfit.c:93,111)"); return MQ_ERR_STATCOR; }
        set_error("a start value could not be drawn inside its bounds after 100000 tries (config lines 9-16, 36-40)");
        return MQ_ERR_RETRY;
    }
    if (status != 0) {
        cudaMemsetAsync(h->solve_status, 0, sizeof(int32_t), h->stream);
        set_error("eikonal solver status %d", status);
        return MQ_ERR_SOLVER;
    }
    return MQ_OK;
}
int check_device_errors(Handle* h)
{
    int32_t flags[2] = {0, 0};
    MQ_CUDA(d2h(&flags[0], h->err, 1, h->stream));
    MQ_CUDA(d2h(&flags[1], h->solve_status, 1, h->stream));
    MQ_CUDA(cudaStreamSynchronize(h->stream));
    h->flags_pending = false;
    return decode_flags(h, flags[0], flags[1]);
}
int flags_enqueue(Handle* h)
{
    MQ_CUDA(d2h(&h->host_flags[0], h->err, 1, h->stream));
    MQ_CUDA(d2h(&h->host_flags[1], h->solve_status, 1, h->stream));
    MQ_CUDA(cudaEventRecord(h->flags_ev, h->stream));
    h->flags_pending = true;
    return MQ_OK;
}
int flags_poll(Handle* h, bool wait)
{
    if (!h->flags_pending) return MQ_OK;
    if (wait) MQ_CUDA(cudaEventSynchronize(h->flags_ev));
    else if (cudaEventQuery(h->flags_ev) != cudaSuccess) { cudaGetLastError(); return MQ_OK; }
    h->flags_pending = false;
    return decode_flags(h, h->host_flags[0], h->host_flags[1]);
}
}  // namespace mq

// forward of the CURRENT state, device side only (no host copies)
namespace mq {
int forward_current_device(Handle* h, int calct)
{
    cudaStream_t s = h->stream;
    sync_cur_view<<<(h->n + 127) / 128, 128, 0, s>>>(h->n, h->mcur, h->tcur, h->ecur, h->cur_view);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    if (h->cfg.aflag == 1) {   // "prior only": all sums are zero, nothing is computed (src/misfit.c:61)
        MQ_CUDA(cudaMemsetAsync(h->mf_eval, 0, 8 * (size_t)h->n * sizeof(float), s));
        MQ_CUDA(cudaMemsetAsync(h->evsum, 0, 2 * (size_t)h->n * h->ne * 8 * sizeof(float), s));
    } else {
        if (calct != 0 && h->cfg.eikonal == 1) {
            const int max_items = h->n * (calct == 3 ? 2 : 1);
            MQ_CUDA(launch_build_items_all(h, h->cur_view, calct));
            MQ_CUDA(launch_rasterise(h, h->cur_view, max_items));
            MQ_CUDA(launch_tables(h, max_items));
        }
        MQ_CUDA(launch_misfit(h, h->cur_view));
        MQ_CUDA(launch_totals(h, h->cur_view));
    }
    adopt_totals_kernel<<<(h->n + 127) / 128, 128, 0, s>>>(h->n, h->sum_of_picks, h->mf_eval, h->noise, h->mf, h->misfit,
                                                            h->rms, h->ll);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    h->forward_done = true;
    return MQ_OK;
}
}  // namespace mq

// ecur_zero: every chain's current event buffer is 0 (right after mq_set_models): no need to ask the device first
static int copy_forward_results(Handle* h, float* mf, float* origin, bool ecur_zero = false)
{
    cudaStream_t s = h->stream;
    const size_t n = h->n;
    if (mf) MQ_CUDA(d2h(mf, h->mf, n * 8, s));
    if (origin && ecur_zero) {
        MQ_CUDA(d2h(origin, h->origin, n * h->ne, s));
    } else if (origin) {
        std::vector<int32_t> ecur(n);
        MQ_CUDA(d2h(ecur.data(), h->ecur, n, s));
        MQ_CUDA(cudaStreamSynchronize(s));
        bool all0 = true;
        for (size_t c = 0; c < n; c++) all0 = all0 && ecur[c] == 0;
        if (all0) MQ_CUDA(d2h(origin, h->origin, n * h->ne, s));
        else
            for (size_t c = 0; c < n; c++)
                MQ_CUDA(d2h(origin + c * h->ne, h->origin + ((size_t)ecur[c] * n + c) * h->ne, h->ne, s));
    }
    return check_device_errors(h);
}

extern "C" int mq_forward(mq_handle* hh, int calct, float* mf, float* origin)
{
    if (!hh || calct < 0 || calct > 3) { set_error("mq_forward: bad argument"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    if (!h->models_set) { set_error("mq_forward: no models in the handle (mq_set_models / mq_init_chains first)"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    const int rc = forward_current_device(h, calct);
    if (rc != MQ_OK) return rc;
    return copy_forward_results(h, mf, origin);
}

extern "C" int mq_forward_host(mq_handle* hh, const mq_models* m, int calct, float* mf, float* origin)
{
    if (!hh || calct < 0 || calct > 3) { set_error("mq_forward_host: bad argument"); return MQ_ERR_ARG; }
    // one pass down the stream: models in, forward, results out, one wait at the end (check_device_errors)
    int rc = set_models(hh, m, false);
    if (rc != MQ_OK) return rc;
    Handle* h = &hh->h;
    rc = forward_current_device(h, calct);
    if (rc != MQ_OK) { cudaStreamSynchronize(h->stream); return rc; }
    return copy_forward_results(h, mf, origin, true);
}

// Host-driven use (a reference-style main that calls mq_forward_host per proposal): the device tables are those of
// the last call with calct != 0.  The reference keeps a backup copy of its tables and restores it after a rejection
// (src/mcmc_eq.c:856,1161,1171); these two calls are that backup / restore, device to device.
static int tables_copy(mq_handle* hh, int from, int to, int phases, const char* who)
{
    if (!hh || phases < 1 || phases > 3) { set_error("%s: bad argument", who); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    if (!h->models_set) { set_error("%s: no models", who); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    const size_t half = (size_t)h->n * 2 * h->tab_stride;
    if (phases == 3) {
        MQ_CUDA(cudaMemcpyAsync(h->tab + (size_t)to * half, h->tab + (size_t)from * half, half * sizeof(float), cudaMemcpyDeviceToDevice,
                                h->stream));
        return MQ_OK;
    }
    // one phase of every chain: rows of tab_stride floats at a pitch of two tables
    const size_t ph = phases == 1 ? 0 : 1, w = h->tab_stride * sizeof(float);
    MQ_CUDA(cudaMemcpy2DAsync(h->tab + (size_t)to * half + ph * h->tab_stride, 2 * w, h->tab + (size_t)from * half + ph * h->tab_stride,
                              2 * w, w, h->n, cudaMemcpyDeviceToDevice, h->stream));
    return MQ_OK;
}
extern "C" int mq_tables_save(mq_handle* hh) { return tables_copy(hh, 0, 1, 3, "mq_tables_save"); }
extern "C" int mq_tables_restore(mq_handle* hh) { return tables_copy(hh, 1, 0, 3, "mq_tables_restore"); }
extern "C" int mq_tables_save_phases(mq_handle* hh, int phases) { return tables_copy(hh, 0, 1, phases, "mq_tables_save_phases"); }
extern "C" int mq_tables_restore_phases(mq_handle* hh, int phases) { return tables_copy(hh, 1, 0, phases, "mq_tables_restore_phases"); }

extern "C" int mq_traveltimet(float* const* ttt, int nx, int ny, int nz, float h, float dist, float z, float z0, float* t_out, int device)
{
    // nx, ny are the grid's horizontal node counts: the distance axis has nxmod = (int)sqrt(nx^2 + ny^2) nodes (src/interpol.c:52)
    if (!ttt || !t_out || nx < 1 || ny < 1 || nz < 2 || !(h > 0.f)) { set_error("mq_traveltimet: bad argument"); return MQ_ERR_ARG; }
    const int nxmod = (int)sqrt((double)(nx * nx + ny * ny));
    int iz1 = 0, m1 = 0;
    if (!traveltimet_cell(dist, z, h, z0, nz, nxmod, &iz1, &m1) || iz1 < 0 || m1 < 0) { *t_out = 1e30f; return MQ_OK; }
    MQ_CUDA(cudaSetDevice(device));
    const float corners[4] = {ttt[iz1][m1], ttt[iz1][m1 + 1], ttt[iz1 + 1][m1], ttt[iz1 + 1][m1 + 1]};
    float* d = nullptr;
    MQ_CUDA(cudaMalloc(&d, 5 * sizeof(float)));
    cudaError_t e = cudaMemcpy(d, corners, sizeof corners, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_traveltimet(dist, z, h, z0, nz, nxmod, d, d + 4, 0);
    if (e == cudaSuccess) e = cudaMemcpy(t_out, d + 4, sizeof(float), cudaMemcpyDeviceToHost);
    cudaFree(d);
    MQ_CUDA(e);
    return MQ_OK;
}

extern "C" int mq_sync(mq_handle* hh)
{
    if (!hh) return MQ_ERR_ARG;
    MQ_CUDA(cudaSetDevice(hh->h.device));
    MQ_CUDA(cudaStreamSynchronize(hh->h.stream));
    return flags_poll(&hh->h, true);
}

extern "C" int mq_get_rows(mq_handle* hh, int chain, int phase, float* rows_out, int32_t* row_index)
{
    if (!hh || chain < 0 || chain >= hh->h.n || (phase != 1 && phase != 2)) { set_error("mq_get_rows: bad argument"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    if (!h->forward_done) { set_error("mq_get_rows: no tables yet (mq_forward first)"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    if (row_index) for (int r = 0; r < h->n_rows; r++) row_index[r] = h->rows_host[r];
    if (rows_out) {
        int32_t tb = 0;
        MQ_CUDA(d2h(&tb, h->tcur + 2 * (size_t)chain + (phase - 1), 1, h->stream));
        MQ_CUDA(cudaStreamSynchronize(h->stream));
        const float* src = h->tab + (((size_t)tb * h->n + chain) * 2 + (phase - 1)) * h->tab_stride;
        std::vector<float> tmp(h->tab_stride);
        MQ_CUDA(d2h(tmp.data(), src, h->tab_stride, h->stream));
        MQ_CUDA(cudaStreamSynchronize(h->stream));
        for (int r = 0; r < h->n_rows; r++)
            for (int k = 0; k < h->nz; k++)
                for (int i = 0; i < h->nxmod; i++)
                    rows_out[((size_t)r * h->nz + k) * h->nxmod + i] = tmp[((size_t)r * h->nz + k) * h->xp + i];
    }
    return h->n_rows;
}

extern "C" int mq_set_tables(mq_handle* hh, int mode)
{
    if (!hh) { set_error("mq_set_tables: null"); return MQ_ERR_ARG; }
    if (mode != MQ_TABLES_PARITY && mode != MQ_TABLES_RECIPROCAL) { set_error("mq_set_tables: mode %d", mode); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    // the tables of the chains in the handle were built in the current mode: it cannot change under them
    if (h->models_set) { set_error("mq_set_tables: call it before mq_set_models / mq_init_chains / mq_state_load"); return MQ_ERR_STATE; }
    h->tables_mode = mode;
    return MQ_OK;
}

extern "C" int mq_get_table(mq_handle* hh, int chain, int phase, float* ttt)
{
    if (!hh || !ttt || chain < 0 || chain >= hh->h.n || (phase != 1 && phase != 2)) { set_error("mq_get_table: bad argument"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    if (h->tables_mode == MQ_TABLES_RECIPROCAL && h->cfg.eikonal == 1 && h->cfg.aflag != 1) {
        set_error("mq_get_table: the handle builds reciprocal tables (mq_set_tables); no parity table exists, mq_get_rows reads the stored rows");
        return MQ_ERR_UNSUPPORTED;
    }
    if (!h->models_set) { set_error("mq_get_table: no models"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int nz = h->nz, nx = h->nxmod;
    const size_t nodes = (size_t)nx * nz;
    // slowness column of (chain, phase) via the regular rasteriser, then a table-mode batch of that one column with full
    // fields: solve g has its source at depth g and its field at d_out + g * nodes
    int32_t one = 1, ph = phase - 1;
    sync_cur_view<<<(h->n + 127) / 128, 128, 0, s>>>(h->n, h->mcur, h->tcur, h->ecur, h->cur_view);
    count_launch();
    MQ_CUDA(h2d(h->n_items, &one, 1, s));
    MQ_CUDA(h2d(h->item_chain, &chain, 1, s));
    MQ_CUDA(h2d(h->item_phase, &ph, 1, s));
    MQ_CUDA(launch_rasterise(h, h->cur_view, 1));
    float* d_out = nullptr;
    MQ_CUDA(cudaMalloc(&d_out, (size_t)nz * nodes * sizeof(float)));
    EikBatch b = {};
    b.nxmod = nx; b.nz = nz; b.slow = h->slow; b.n_items = 1;
    b.full_out = d_out; b.status_min = h->solve_status;
    std::vector<float> t((size_t)nz * nodes);
    cudaError_t e = eik_launch(b, h->eik, s);
    if (e == cudaSuccess) e = d2h(t.data(), d_out, t.size(), s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFree(d_out);
    MQ_CUDA(e);
    // ttt[j][iz][i] = t_iz[i*nz + j]   (src/misfit.c:281-288)
    for (int j = 0; j < nz; j++)
        for (int k = 0; k < nz; k++)
            for (int i = 0; i < nx; i++) ttt[((size_t)j * nz + k) * nx + i] = t[(size_t)k * nodes + (size_t)i * nz + j];
    return check_device_errors(h);
}

extern "C" int mq_get_predictions(mq_handle* hh, int chain, float* resid, float* tpred)
{
    if (!hh || chain < 0 || chain >= hh->h.n) { set_error("mq_get_predictions: bad argument"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    if (!h->models_set) { set_error("mq_get_predictions: no models"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    if (!h->tpred) MQ_CUDA(cudaMalloc(&h->tpred, (size_t)h->n * h->np * sizeof(float)));
    // re-run the residual loop on the current tables with per-pick output switched on
    h->want_pred = true;
    sync_cur_view<<<(h->n + 127) / 128, 128, 0, h->stream>>>(h->n, h->mcur, h->tcur, h->ecur, h->cur_view);
    count_launch();
    cudaError_t e = launch_misfit(h, h->cur_view);
    h->want_pred = false;
    MQ_CUDA(e);
    if (resid) MQ_CUDA(d2h(resid, h->resid + (size_t)chain * h->np, h->np, h->stream));
    if (tpred) MQ_CUDA(d2h(tpred, h->tpred + (size_t)chain * h->np, h->np, h->stream));
    MQ_CUDA(cudaStreamSynchronize(h->stream));
    return check_device_errors(h);
}

extern "C" int mq_profile(mq_handle* hh, int enable, double* eikonal_ms, int64_t* eikonal_launches, int64_t* solves_per_full_launch)
{
    if (!hh) { set_error("mq_profile: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    MQ_CUDA(cudaSetDevice(h->device));
    double ms = 0;
    long n = 0;
    profile_collect(h, &ms, &n, enable != 0);
    profile_enable(h, enable != 0);
    if (eikonal_ms) *eikonal_ms = ms;
    if (eikonal_launches) *eikonal_launches = n;
    if (solves_per_full_launch)
        *solves_per_full_launch = (int64_t)2 * h->n * (h->tables_mode == MQ_TABLES_RECIPROCAL ? h->n_rows : h->nz);
    return MQ_OK;
}

extern "C" int mq_profile_kernels(mq_handle* hh, int64_t* launches, double* ms)
{
    if (!hh) { set_error("mq_profile_kernels: null"); return MQ_ERR_ARG; }
    double m[kEikKernels]; long n[kEikKernels];
    profile_by_kernel(&hh->h, m, n);
    for (int k = 0; k < kEikKernels; k++) { if (launches) launches[k] = n[k]; if (ms) ms[k] = m[k]; }
    return MQ_OK;
}
extern "C" const char* mq_eikonal_kernel_name(int k) { return eik_kernel_name(k); }
extern "C" int mq_profile_misfit(mq_handle* hh, int64_t* launches, double* ms)
{
    if (!hh) { set_error("mq_profile_misfit: null"); return MQ_ERR_ARG; }
    double m = 0; long n = 0;
    profile_misfit(&hh->h, &m, &n);
    if (launches) *launches = n;
    if (ms) *ms = m;
    return MQ_OK;
}

// ---- device timers on the handle's stream (bench.py times K steps with these) ---------------------
extern "C" int mq_timer(mq_handle* hh, int slot, int stop, double* elapsed_ms)
{
    if (!hh || slot < 0 || slot >= 16) { set_error("mq_timer: bad argument"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    MQ_CUDA(cudaSetDevice(h->device));
    cudaEvent_t& e = h->timer_ev[stop ? 1 : 0][slot];
    if (!e) MQ_CUDA(cudaEventCreate(&e));
    MQ_CUDA(cudaEventRecord(e, h->stream));
    if (stop) {
        MQ_CUDA(cudaEventSynchronize(e));
        float ms = 0.f;
        if (!h->timer_ev[0][slot]) { set_error("mq_timer: stop without start"); return MQ_ERR_STATE; }
        MQ_CUDA(cudaEventElapsedTime(&ms, h->timer_ev[0][slot], e));
        if (elapsed_ms) *elapsed_ms = ms;
    }
    return MQ_OK;
}
