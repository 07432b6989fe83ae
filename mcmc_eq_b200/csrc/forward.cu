// forward.cu -- rasterise + travel-time lookup + residual/misfit kernels (sm_100a).
//
// Reference: setup_table_new's rasteriser (src/misfit.c:205-266), traveltimet
// (src/interpol.c:43-83), dst (src/mcmc_eq.c:1303-1306) and the residual loop of
// cal_fit_newx (src/misfit.c:83-153), for all chains at once.
#include "forward.cuh"
#include "eikonal.cuh"
#include "launch_count.h"
#include "tria.cuh"

#include <stdlib.h>
#include <vector>

namespace mq {

// ---- work list for "all chains" ---------------------------------------------------------
__global__ void build_items_all_kernel(int n, int calct, size_t tab_stride, float* tab, const int32_t* tbuf,
                                       int32_t* item_chain, int32_t* item_phase, float** item_tab, int32_t* n_items)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int per = (calct == 3) ? 2 : 1;
    if (c == 0) *n_items = n * per;
    if (c >= n) return;
    int k = 0;
    for (int ph = 0; ph < 2; ph++) {
        if (!(calct & (1 << ph))) continue;
        const int item = c * per + k++;
        item_chain[item] = c;
        item_phase[item] = ph;
        item_tab[item] = tab + (((size_t)tbuf[2 * c + ph] * n + c) * 2 + ph) * tab_stride;
    }
}

cudaError_t launch_build_items_all(Handle* h, const EvalView& v, int calct)
{
    build_items_all_kernel<<<(h->n + 127) / 128, 128, 0, h->stream>>>(h->n, calct, h->tab_stride, h->tab, v.tbuf,
                                                                      h->item_chain, h->item_phase, h->item_tab, h->n_items);
    count_launch();
    return cudaGetLastError();
}

// ---- Voronoi rasteriser -------------------------------------------------------------------
// One thread per (item, depth node).  Nearest nucleus in depth, ties -> highest index
// (find_in_cell, src/mod_grd.c:93-110); vs = vp/vpvs; slow = h/v (src/misfit.c:209-213,263).
// tria != 0: linear interpolation between the depth-sorted nuclei instead (src/misfit.c:217-250, tria.cuh).
__global__ void rasterise_kernel(int nz, int md, int n, float hgrid, float z0, int tria, const int32_t* n_items,
                                 const int32_t* item_chain, const int32_t* item_phase, const int32_t* mbuf,
                                 const int32_t* dim, const float* z, const float* vp, const float* vpvs, float* slow)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int item = t / nz, iz = t - item * nz;
    if (item >= *n_items) return;
    const int c = item_chain[item];
    const int b = mbuf[c];
    const size_t mo = ((size_t)b * n + c) * md;
    const int d = dim[b * n + c];
    if (tria) {
        int lo, hi;
        tria::segment_of_node(z + mo, d, iz, hgrid, z0, &lo, &hi);
        const float zq = __fadd_rn(z0, __fmul_rn((float)iz, hgrid));
        const bool isS = item_phase[item] != 0;
        const float v0 = isS ? __fdiv_rn(vp[mo + lo], vpvs[mo + lo]) : vp[mo + lo];
        const float v1 = isS ? __fdiv_rn(vp[mo + hi], vpvs[mo + hi]) : vp[mo + hi];
        slow[(size_t)item * nz + iz] = __fdiv_rn(hgrid, tria::line_through(zq, z[mo + lo], v0, z[mo + hi], v1));
        return;
    }
    const float zq = __fadd_rn(z0, __fmul_rn((float)iz, hgrid));
    float best = 3.402823466e+38f;
    int k = 0;
    for (int i = 0; i < d; i++) {
        const float dz = __fsub_rn(z[mo + i], zq);
        const float d2 = __fmul_rn(dz, dz);
        if (d2 <= best) { best = d2; k = i; }
    }
    const float p = vp[mo + k];
    const float v = item_phase[item] == 0 ? p : __fdiv_rn(p, vpvs[mo + k]);
    slow[(size_t)item * nz + iz] = __fdiv_rn(hgrid, v);
}

cudaError_t launch_rasterise(Handle* h, const EvalView& v, int max_items)
{
    const int threads = max_items * h->nz;
    if (threads <= 0) return cudaSuccess;
    rasterise_kernel<<<(threads + 127) / 128, 128, 0, h->stream>>>(h->nz, h->md, h->n, h->cfg.grid.h, h->cfg.grid.z0, h->cfg.tria,
                                                                    h->n_items, h->item_chain, h->item_phase, v.mbuf, h->dim,
                                                                    h->z, h->vp, h->vpvs, h->slow);
    count_launch();
    return cudaGetLastError();
}

// ---- timing of the eikonal launches (mq_profile) -------------------------------------------
struct Profile {
    std::vector<cudaEvent_t> ev;   // start/stop pairs not yet read
    std::vector<int> which;        // kernel each pair's launch took (eikonal.cuh: kEik*)
    double ms_total = 0;
    long launches = 0;
    double ms_by[kEikKernels] = {0, 0, 0, 0};
    long n_by[kEikKernels] = {0, 0, 0, 0};
    std::vector<cudaEvent_t> mev;  // start/stop pairs round the misfit kernel
    double misfit_ms = 0, misfit_ms_read = 0;
    long misfit_n = 0, misfit_n_read = 0;
    bool enabled = false;
};

void profile_enable(Handle* h, bool on)
{
    if (!h->prof) h->prof = new Profile();
    ((Profile*)h->prof)->enabled = on;
}
void profile_collect(Handle* h, double* ms, long* launches, bool reset)
{
    Profile* p = (Profile*)h->prof;
    if (!p) { *ms = 0; *launches = 0; return; }
    for (size_t i = 0; i + 1 < p->ev.size(); i += 2) {
        float t = 0.f;
        cudaEventSynchronize(p->ev[i + 1]);
        cudaEventElapsedTime(&t, p->ev[i], p->ev[i + 1]);
        p->ms_total += t;
        p->launches++;
        const int w = p->which[i / 2];
        p->ms_by[w] += t;
        p->n_by[w]++;
        cudaEventDestroy(p->ev[i]);
        cudaEventDestroy(p->ev[i + 1]);
    }
    p->ev.clear();
    p->which.clear();
    for (size_t i = 0; i + 1 < p->mev.size(); i += 2) {
        float t = 0.f;
        cudaEventSynchronize(p->mev[i + 1]);
        cudaEventElapsedTime(&t, p->mev[i], p->mev[i + 1]);
        p->misfit_ms += t;
        p->misfit_n++;
        cudaEventDestroy(p->mev[i]);
        cudaEventDestroy(p->mev[i + 1]);
    }
    p->mev.clear();
    *ms = p->ms_total;
    *launches = p->launches;
    if (reset) {
        p->ms_total = 0; p->launches = 0;
        for (int k = 0; k < kEikKernels; k++) { p->ms_by[k] = 0; p->n_by[k] = 0; }
        p->misfit_ms_read = p->misfit_ms; p->misfit_n_read = p->misfit_n;
        p->misfit_ms = 0; p->misfit_n = 0;
    } else {
        p->misfit_ms_read = p->misfit_ms; p->misfit_n_read = p->misfit_n;
    }
}
void profile_misfit(Handle* h, double* ms, long* launches)
{
    Profile* p = (Profile*)h->prof;
    *ms = p ? p->misfit_ms_read : 0.0;
    *launches = p ? p->misfit_n_read : 0;
}
void profile_by_kernel(Handle* h, double* ms, long* launches)
{
    Profile* p = (Profile*)h->prof;
    for (int k = 0; k < kEikKernels; k++) { ms[k] = p ? p->ms_by[k] : 0.0; launches[k] = p ? p->n_by[k] : 0; }
}
void profile_destroy(Handle* h)
{
    double a; long b;
    if (h->prof) { profile_collect(h, &a, &b, true); delete (Profile*)h->prof; h->prof = nullptr; }
}

cudaError_t launch_tables(Handle* h, int max_items)
{
    Profile* pr = (Profile*)h->prof;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (pr && pr->enabled) {
        cudaEventCreate(&e0); cudaEventCreate(&e1);
        cudaEventRecord(e0, h->stream);
    }
    int which = kEikGeneric;
    struct Stop {
        Profile* pr; cudaEvent_t e0, e1; cudaStream_t s; int* which;
        ~Stop() { if (e0) { cudaEventRecord(e1, s); pr->ev.push_back(e0); pr->ev.push_back(e1); pr->which.push_back(*which); } }
    } stop{pr, e0, e1, h->stream, &which};
    EikBatch b = {};
    b.nxmod = h->nxmod; b.nz = h->nz;
    b.slow = h->slow; b.n_items = max_items; b.n_items_dev = h->n_items;
    b.row_out = h->item_tab; b.rows = h->d_rows; b.n_rows = h->n_rows; b.xpitch = h->xp;
    if (h->tables_mode == MQ_TABLES_RECIPROCAL) {
        // sources at the receiver rows, every row of their fields kept
        b.src_rows = h->d_rows; b.n_src_rows = h->n_rows;
        b.rows = h->d_all_rows; b.n_rows = h->nz;
    }
    b.status_min = h->solve_status;
    b.regroup = true;
    return eik_launch(b, h->eik, h->stream, &which);
}

// ---- travel-time lookup -------------------------------------------------------------------
// Bilinear interpolation of (dist, z) in a [nz][xp] receiver-row table; the same arithmetic as traveltimet
// (src/interpol.c:56-80): float corner products summed left to right, the 1/(dx*dy) prefactor in double.  The depth part
// is the same for every pick of an event and is set up once per warp; 1/(x2-x1)/(y2-y1) is only divided out per pick when
// the float difference x2-x1 is not the grid spacing itself (never for a power-of-two spacing).
struct BilinearZ {
    int iz1;
    float c, d, dyf;    // y2-y, y-y1, y2-y1
    double pref0;       // 1 / h / (y2-y1)
    bool oob;
};

__device__ __forceinline__ BilinearZ bilinear_depth(float z, float hgrid, float z0, int nz)
{
    BilinearZ w;
    const float y = __fsub_rn(z, z0);
    w.iz1 = (int)__fdiv_rn(y, hgrid);
    w.oob = w.iz1 >= nz - 1;
    const float y1 = __fmul_rn((float)w.iz1, hgrid), y2 = __fmul_rn((float)(w.iz1 + 1), hgrid);
    w.c = __fsub_rn(y2, y);
    w.d = __fsub_rn(y, y1);
    w.dyf = __fsub_rn(y2, y1);
    w.pref0 = 1.0 / (double)hgrid / (double)w.dyf;
    return w;
}

struct BilinearX {
    int m1;
    float a, b;         // x2-x, x-x1
    double pref;
    bool oob;
};

// rh = 1/hgrid, used instead of the division when hgrid is a power of two (bit-identical then)
__device__ __forceinline__ BilinearX bilinear_dist(const BilinearZ& wz, float dist, float hgrid, float rh, bool h_pow2, int nxmod)
{
    BilinearX w;
    w.m1 = (int)(h_pow2 ? __fmul_rn(dist, rh) : __fdiv_rn(dist, hgrid));
    w.oob = wz.oob || w.m1 >= nxmod - 1;
    const float x1 = __fmul_rn((float)w.m1, hgrid), x2 = __fmul_rn((float)(w.m1 + 1), hgrid);
    w.a = __fsub_rn(x2, dist);
    w.b = __fsub_rn(dist, x1);
    const float dxf = __fsub_rn(x2, x1);
    w.pref = (dxf == hgrid) ? wz.pref0 : 1.0 / (double)dxf / (double)wz.dyf;
    return w;
}

// row: the [nz][xp] table of one receiver row, already offset to depth row iz1
__device__ __forceinline__ float bilinear_eval(const BilinearZ& wz, const BilinearX& w, const float* __restrict__ row, int xp)
{
    const float* p = row + w.m1;
    const float v1 = __ldg(p), v2 = __ldg(p + 1), v3 = __ldg(p + xp), v4 = __ldg(p + xp + 1);
    float s = __fmul_rn(__fmul_rn(v1, w.a), wz.c);
    s = __fadd_rn(s, __fmul_rn(__fmul_rn(v2, w.b), wz.c));
    s = __fadd_rn(s, __fmul_rn(__fmul_rn(v3, w.a), wz.d));
    s = __fadd_rn(s, __fmul_rn(__fmul_rn(v4, w.b), wz.d));
    return (float)(w.pref * (double)s);
}

// One lookup with the four corner values handed in (mq_traveltimet): corners = t[iz1][m1], t[iz1][m1+1], t[iz1+1][m1], t[iz1+1][m1+1]
__global__ void traveltimet_kernel(float dist, float z, float hgrid, float z0, int nz, int nxmod, const float* corners, float* out)
{
    const BilinearZ wz = bilinear_depth(z, hgrid, z0, nz);
    const BilinearX w = bilinear_dist(wz, dist, hgrid, 1.0f / hgrid, false, nxmod);
    if (w.oob) { *out = 1e30f; return; }
    BilinearX w0 = w;
    w0.m1 = 0;
    *out = bilinear_eval(wz, w0, corners, 2);
}

// cell the lookup of (dist, z) reads, computed on the host with the same float operations (src/interpol.c:56-63)
bool traveltimet_cell(float dist, float z, float hgrid, float z0, int nz, int nxmod, int* iz1, int* m1)
{
    const float y = z - z0;
    *iz1 = (int)(y / hgrid);
    *m1 = (int)(dist / hgrid);
    return !(*iz1 >= nz - 1 || *m1 >= nxmod - 1);
}

cudaError_t launch_traveltimet(float dist, float z, float hgrid, float z0, int nz, int nxmod, const float* d_corners, float* d_out,
                               cudaStream_t s)
{
    traveltimet_kernel<<<1, 1, 0, s>>>(dist, z, hgrid, z0, nz, nxmod, d_corners, d_out);
    count_launch();
    return cudaGetLastError();
}

__device__ __forceinline__ float warp_sum(float v)
{
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- residuals / origin time / class sums --------------------------------------------------
// One warp per (chain, event): lanes stride over the event's picks (P first, then S).  The event's residuals never leave
// the SM: lane l keeps the raw residuals of picks l, l + 32, ... in its column of a per-warp strip of shared memory
// (kMisfitKeep of them: an event of config 3 / 4 has 100 / 200 picks = 4 / 7 per lane), takes part in the warp sum that
// gives the origin time (src/misfit.c:121-123), de-means its own and adds the squares to the eight class sums
// (src/misfit.c:146-153), which live in a second strip indexed by class (one read-modify-write per pick instead of eight
// selects).  Per-pick values reach HBM only when mq_get_predictions asks for them (want_pred).
// Events with more than 32 * kMisfitKeep picks take the same kernel with the residuals in a global scratch (KEEP == false).
// With a power-of-two grid spacing every bilinear prefactor 1 / ((x2-x1)(y2-y1)) is a power of two, so the reference's
// double product (src/interpol.c:80) equals a float product bit for bit and no FP64 instruction is issued.
struct MisfitParams {
    int n, ne, ns, np, nz, nxmod, xp, md;
    float hgrid, z0, rh;
    int eikonal, scor_flag, h_pow2;
    size_t tab_stride;
    DevPicks pk;
    EvalView v;
    const int32_t* dim;
    const float *z, *vp, *vpvs;
    const float *eq, *pres, *sres;
    const float* tab;
    float *evsum, *origin, *evq, *oq;
    float *resid, *tpred;
    int32_t* err;
};

constexpr int kMisfitWarps = 4;
constexpr int kMisfitKeep = 8;      // residuals per lane kept in shared memory: events of up to 256 picks

// KEEP: residuals stay in shared memory; POW2: power-of-two grid spacing (float prefactor, no division); RAY: the
// straight-ray branch eikonal == 0 (src/misfit.c:90,108) instead of the table lookup.
template <bool KEEP, bool POW2, bool RAY>
__global__ void __launch_bounds__(kMisfitWarps * 32, 8) misfit_kernel(MisfitParams p)
{
    __shared__ float class_acc[kMisfitWarps][8][32];
    __shared__ float res_keep[KEEP ? kMisfitWarps : 1][KEEP ? kMisfitKeep : 1][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long task = (long)blockIdx.x * kMisfitWarps + wib;
    if (task >= (long)p.n * p.ne) return;
    const int c = (int)(task / p.ne), e = (int)(task - (long)c * p.ne);
    if (p.v.hold && p.v.hold[c] != 0) return;
    const int only = p.v.ev_only[c];
    if (only == -2 || (only >= 0 && only != e)) return;

    float ex, ey, ez;
    if (p.v.q_idx[c] == e) { ex = p.v.q_xyz[3 * c]; ey = p.v.q_xyz[3 * c + 1]; ez = p.v.q_xyz[3 * c + 2]; }
    else { const float* q = p.eq + ((size_t)c * p.ne + e) * 3; ex = q[0]; ey = q[1]; ez = q[2]; }

    // proposed station-correction perturbation (src/mcmc_eq.c:910-928), the same for every pick of the chain: the
    // chosen station gets +d1 (and +d2 under a non-zero scor_flag), every other one -d1/(nos-1) when scor_flag <= 0
    const int ridx = p.v.r_idx[c];
    float rd1P = 0.f, rd1S = 0.f, rd2P = 0.f, rd2S = 0.f, rq1P = 0.f, rq1S = 0.f;
    if (ridx >= 0) {
        const float* rd = p.v.r_d + 4 * (size_t)c;
        const float nsm1 = (float)(p.ns - 1);
        rd1P = rd[0]; rd1S = rd[1]; rd2P = rd[2]; rd2S = rd[3];
        rq1P = __fdiv_rn(rd1P, nsm1); rq1S = __fdiv_rn(rd1S, nsm1);
    }
    const float* pres = (ridx == -2) ? p.v.pres_over + (size_t)c * p.ns : p.pres + (size_t)c * p.ns;
    const float* sres = (ridx == -2) ? p.v.sres_over + (size_t)c * p.ns : p.sres + (size_t)c * p.ns;

    const int b = p.pk.ev_off[e], end = p.pk.ev_off[e + 1], npk = p.pk.n_p[e];
    const int rowsz = p.nz * p.xp;      // a (chain, phase) table holds n_rows * nz * xp floats: 32-bit offsets inside it
    float* resid = (!KEEP || p.tpred) ? p.resid + (size_t)c * p.np : nullptr;

    float v0p = 1.f, v0s = 1.f;
    BilinearZ wz;
    wz.iz1 = 0; wz.c = wz.d = wz.dyf = 0.f; wz.pref0 = 0.0; wz.oob = false;
    if (RAY) {   // velocity of the nucleus nearest to z = 0
        const int mb = p.v.mbuf[c];
        const size_t mo = ((size_t)mb * p.n + c) * p.md;
        const int d = p.dim[mb * p.n + c];
        float best = 3.402823466e+38f;
        int k = 0;
        for (int i = 0; i < d; i++) {
            const float d2 = __fmul_rn(p.z[mo + i], p.z[mo + i]);
            if (d2 <= best) { best = d2; k = i; }
        }
        v0p = p.vp[mo + k];
        v0s = __fdiv_rn(v0p, p.vpvs[mo + k]);
    } else if (POW2) {   // depth part of the bilinear weights; y / h == y * (1/h) and every product below is exact
        const float y = __fsub_rn(ez, p.z0);
        wz.iz1 = (int)__fmul_rn(y, p.rh);
        wz.oob = wz.iz1 >= p.nz - 1;
        wz.c = __fsub_rn(__fmul_rn((float)(wz.iz1 + 1), p.hgrid), y);
        wz.d = __fsub_rn(y, __fmul_rn((float)wz.iz1, p.hgrid));
    } else {
        wz = bilinear_depth(ez, p.hgrid, p.z0, p.nz);
    }
    const float pref0f = p.rh * p.rh;     // POW2: 1 / ((x2-x1)(y2-y1)) = 1/h^2 exactly (src/interpol.c:80)
    const int zoff = (wz.oob ? 0 : wz.iz1) * p.xp;
    const float* tabPz = p.tab + (((size_t)p.v.tbuf[2 * c] * p.n + c) * 2 + 0) * p.tab_stride + zoff;
    const float* tabSz = p.tab + (((size_t)p.v.tbuf[2 * c + 1] * p.n + c) * 2 + 1) * p.tab_stride + zoff;
    float sum = 0.f;
    bool oob = false;         // a pick fell outside the table (1e30 sentinel of src/interpol.c:64-65)
    float* keep_l = &res_keep[KEEP ? wib : 0][0][lane];     // raw residual of this lane's i-th pick at keep_l[32 i]

    // the pick's constants in two vector loads: (x, y, t, w1) and (w2, station | row << 20 | class << 28)
    auto one_pick = [&](int j) -> float {
        const int isS = ((j - b) >= npk) ? 1 : 0;
        const float4 r4 = __ldg(p.pk.rec4 + j);
        const float2 r2 = __ldg(p.pk.rec2 + j);
        const unsigned code = __float_as_uint(r2.y);
        const int st = (int)(code & 0xfffffu), r0 = (int)((code >> 20) & 0xffu);
        float corr = isS ? sres[st] : pres[st];
        const float dx = __fsub_rn(r4.x, ex), dy = __fsub_rn(r4.y, ey);
        const float dist = sqrtf(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
        float tt;
        if (RAY) {
            const float r2 = __fadd_rn(__fmul_rn(dist, dist), __fmul_rn(ez, ez));
            tt = (float)(sqrt((double)r2) / (double)(isS ? v0s : v0p));
        } else if (POW2) {
            const int m1 = (int)__fmul_rn(dist, p.rh);
            const bool out = wz.oob || m1 >= p.nxmod - 1;
            oob = oob || out;
            const float wa = __fsub_rn(__fmul_rn((float)(m1 + 1), p.hgrid), dist), wb = __fsub_rn(dist, __fmul_rn((float)m1, p.hgrid));
            const float* q = (isS ? tabSz : tabPz) + (r0 * rowsz + (out ? 0 : m1));
            float t12[2];
#pragma unroll
            for (int r = 0; r < 2; r++, q += rowsz) {
                const float v1 = __ldg(q), v2 = __ldg(q + 1), v3 = __ldg(q + p.xp), v4 = __ldg(q + p.xp + 1);
                float s4 = __fmul_rn(__fmul_rn(v1, wa), wz.c);
                s4 = __fadd_rn(s4, __fmul_rn(__fmul_rn(v2, wb), wz.c));
                s4 = __fadd_rn(s4, __fmul_rn(__fmul_rn(v3, wa), wz.d));
                s4 = __fadd_rn(s4, __fmul_rn(__fmul_rn(v4, wb), wz.d));
                t12[r] = out ? 1e30f : __fmul_rn(pref0f, s4);
            }
            tt = __fadd_rn(__fmul_rn(t12[0], r4.w), __fmul_rn(t12[1], r2.x));
        } else {
            const BilinearX w = bilinear_dist(wz, dist, p.hgrid, p.rh, false, p.nxmod);
            oob = oob || w.oob;
            const float* row = (isS ? tabSz : tabPz) + r0 * rowsz;
            const float t1 = w.oob ? 1e30f : bilinear_eval(wz, w, row, p.xp);
            const float t2 = w.oob ? 1e30f : bilinear_eval(wz, w, row + rowsz, p.xp);
            tt = __fadd_rn(__fmul_rn(t1, r4.w), __fmul_rn(t2, r2.x));
        }
        if (ridx >= 0) {
            const bool self = st == ridx;
            if (p.scor_flag <= 0) corr = self ? __fadd_rn(corr, isS ? rd1S : rd1P) : __fsub_rn(corr, isS ? rq1S : rq1P);
            if (p.scor_flag != 0 && self) corr = __fadd_rn(corr, isS ? rd2S : rd2P);
        }
        if (corr < -1000.f) atomicOr(p.err, kErrStatcor);
        tt = __fadd_rn(tt, corr);
        if (p.tpred) p.tpred[(size_t)c * p.np + j] = tt;
        return __fsub_rn(tt, r4.z);
    };

#pragma unroll 2
    for (int j = b + lane, i = 0; j < end; j += 32, i++) {
        const float diff = one_pick(j);
        if (KEEP) keep_l[32 * i] = diff;
        else resid[j] = diff;
        sum += diff;
    }
    sum = warp_sum(sum);
    const float mean = sum / (float)(end - b);
    __syncwarp();

    float* acc_l = &class_acc[wib][0][lane];
#pragma unroll
    for (int k = 0; k < 8; k++) acc_l[k * 32] = 0.f;
    for (int j = b + lane, i = 0; j < end; j += 32, i++) {
        const float d = __fsub_rn(KEEP ? keep_l[32 * i] : resid[j], mean);
        if (p.tpred) resid[j] = d;
        acc_l[p.pk.cp[j] * 32] += d * d;
    }
    // The eight class sums over the warp by recursive halving: at every step a lane hands the half of its values that its
    // partner carries on with to that partner (8 -> 4 -> 2 -> 1 values per lane: 7 shuffles), two more steps sum the one value
    // left over the four lanes that share it: 9 shuffles instead of 40.  Lane l ends up with the sum of class
    // 4 * bit4(l) + 2 * bit3(l) + bit2(l); the order of the additions is fixed, so the sums are deterministic.
    float cls_sum;
    const int cls = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
    {
        float v[8], w4[4], w2v[2];
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = acc_l[k * 32];
        const bool hi16 = lane & 16, hi8 = lane & 8, hi4 = lane & 4;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const float give = hi16 ? v[k] : v[k + 4];
            w4[k] = (hi16 ? v[k + 4] : v[k]) + __shfl_xor_sync(0xffffffffu, give, 16);
        }
#pragma unroll
        for (int k = 0; k < 2; k++) {
            const float give = hi8 ? w4[k] : w4[k + 2];
            w2v[k] = (hi8 ? w4[k + 2] : w4[k]) + __shfl_xor_sync(0xffffffffu, give, 8);
        }
        const float give = hi4 ? w2v[0] : w2v[1];
        cls_sum = (hi4 ? w2v[1] : w2v[0]) + __shfl_xor_sync(0xffffffffu, give, 4);
        cls_sum += __shfl_xor_sync(0xffffffffu, cls_sum, 2);
        cls_sum += __shfl_xor_sync(0xffffffffu, cls_sum, 1);
    }
    // With a 1e30 prediction in the event every de-meaned residual of it is ~1e29 or more and its
    // square overflows FP32 in the reference: the event's classes get an infinite misfit.  Stated
    // explicitly here because the overflow would otherwise depend on the summation order.
    if (__any_sync(0xffffffffu, oob)) {
        unsigned present = 0u;    // classes that occur in this event
        for (int j = b + lane; j < end; j += 32) present |= 1u << p.pk.cp[j];
        present = __reduce_or_sync(0xffffffffu, present);
        if (present & (1u << cls)) cls_sum = __int_as_float(0x7f800000);
    }
    if ((lane & 3) == 0) {      // one lane per class
        if (only >= 0) {
            p.evq[8 * (size_t)c + cls] = cls_sum;
            if (lane == 0) p.oq[c] = -mean;
        } else {
            const int eb = p.v.ebuf[c];
            p.evsum[(((size_t)eb * p.n + c) * p.ne + e) * 8 + cls] = cls_sum;
            if (lane == 0) p.origin[((size_t)eb * p.n + c) * p.ne + e] = -mean;
        }
    }
}

cudaError_t launch_misfit(Handle* h, const EvalView& v)
{
    MisfitParams p;
    p.n = h->n; p.ne = h->ne; p.ns = h->ns; p.np = h->np; p.nz = h->nz; p.nxmod = h->nxmod; p.xp = h->xp; p.md = h->md;
    p.hgrid = h->cfg.grid.h; p.z0 = h->cfg.grid.z0; p.rh = 1.0f / p.hgrid;
    // MCMCEQ_MISFIT_POW2=0: the general instantiation for every spacing (checks that the power-of-two one is bit-identical)
    static int allow_pow2 = -1;
    if (allow_pow2 < 0) { const char* e = getenv("MCMCEQ_MISFIT_POW2"); allow_pow2 = (e && e[0] == '0') ? 0 : 1; }
    { int ex = 0; p.h_pow2 = (allow_pow2 && p.hgrid > 0.f && frexpf(p.hgrid, &ex) == 0.5f) ? 1 : 0; }
    p.eikonal = h->cfg.eikonal; p.scor_flag = h->cfg.scor_flag;
    p.tab_stride = h->tab_stride; p.pk = h->pk; p.v = v; p.dim = h->dim; p.z = h->z; p.vp = h->vp; p.vpvs = h->vpvs;
    p.eq = h->eq; p.pres = h->pres; p.sres = h->sres; p.tab = h->tab; p.evsum = h->evsum; p.origin = h->origin;
    p.evq = h->evq; p.oq = h->oq; p.resid = h->resid; p.tpred = h->want_pred ? h->tpred : nullptr; p.err = h->err;
    const long tasks = (long)h->n * h->ne;
    const unsigned grid = (unsigned)((tasks + kMisfitWarps - 1) / kMisfitWarps);
    const int per_lane = (h->pk.max_event_picks + 31) / 32;
    // the per-pick scratch exists when an event is too large for the register path or predictions are wanted
    if ((per_lane > kMisfitKeep || h->want_pred) && !h->resid) {
        const cudaError_t e = cudaMalloc(&h->resid, (size_t)h->n * h->np * sizeof(float));
        if (e != cudaSuccess) return e;
        p.resid = h->resid;
    }
#define MISFIT_LAUNCH(KEEP)                                                                            \
    do {                                                                                               \
        if (p.eikonal == 0) misfit_kernel<KEEP, false, true><<<grid, kMisfitWarps * 32, 0, h->stream>>>(p);        \
        else if (p.h_pow2) misfit_kernel<KEEP, true, false><<<grid, kMisfitWarps * 32, 0, h->stream>>>(p);         \
        else misfit_kernel<KEEP, false, false><<<grid, kMisfitWarps * 32, 0, h->stream>>>(p);                      \
    } while (0)
    static int force_scratch = -1;      // MCMCEQ_MISFIT_SCRATCH=1: residuals through the global scratch (the round-1 data flow)
    if (force_scratch < 0) { const char* e = getenv("MCMCEQ_MISFIT_SCRATCH"); force_scratch = (e && e[0] == '1') ? 1 : 0; }
    if (force_scratch && !h->resid) {
        const cudaError_t e = cudaMalloc(&h->resid, (size_t)h->n * h->np * sizeof(float));
        if (e != cudaSuccess) return e;
        p.resid = h->resid;
    }
    Profile* pr = (Profile*)h->prof;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (pr && pr->enabled) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, h->stream); }
    if (per_lane <= kMisfitKeep && !force_scratch) MISFIT_LAUNCH(true);
    else MISFIT_LAUNCH(false);
#undef MISFIT_LAUNCH
    if (e0) { cudaEventRecord(e1, h->stream); pr->mev.push_back(e0); pr->mev.push_back(e1); }
    count_launch();
    return cudaGetLastError();
}

// ---- per-chain totals -----------------------------------------------------------------------
// One warp per chain; double accumulation over events in a fixed order (deterministic).
__global__ void __launch_bounds__(128) totals_kernel(int n, int ne, EvalView v, const int32_t* ecur, const float* evsum,
                                                     const float* evq, const float* mf_cur, float* mf_eval)
{
    const int lane = threadIdx.x & 31;
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (c >= n) return;
    if (v.hold && v.hold[c] != 0) return;
    const int only = v.ev_only[c];
    if (only == -2) {   // nothing re-evaluated (noise proposal): the sums are those of the current model
        if (lane < 8) mf_eval[8 * (size_t)c + lane] = mf_cur[8 * (size_t)c + lane];
        return;
    }
    const int eb = (only >= 0) ? ecur[c] : v.ebuf[c];
    const float* src = evsum + ((size_t)eb * n + c) * ne * 8;
    double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int e = lane; e < ne; e += 32) {
        const float* s = (e == only) ? evq + 8 * (size_t)c : src + (size_t)e * 8;
#pragma unroll
        for (int k = 0; k < 8; k++) acc[k] += (double)s[k];
    }
#pragma unroll
    for (int k = 0; k < 8; k++)
        for (int o = 16; o; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    if (lane == 0)
        for (int k = 0; k < 8; k++) mf_eval[8 * (size_t)c + k] = (float)acc[k];
}

cudaError_t launch_totals(Handle* h, const EvalView& v)
{
    const int wpb = 4;
    totals_kernel<<<(h->n + wpb - 1) / wpb, wpb * 32, 0, h->stream>>>(h->n, h->ne, v, h->ecur, h->evsum, h->evq, h->mf,
                                                                       h->mf_eval);
    count_launch();
    return cudaGetLastError();
}

}  // namespace mq
