// chain.cu -- batched transdimensional Metropolis-Hastings step on the device.
//
// Reference: the main loop of mcmc_eq (src/mcmc_eq.c:845-1192): proposal arms Q,R,P,V,M,B,D,N,
// model_valid (:180-229), rand_* helpers (:122-178), start model (:559-630), acceptance
// (:1135-1164).  One thread per chain draws the proposal from a counter-based RNG
// (Philox4x32-10 keyed by seed, indexed by chain and draw number), the forward kernels
// evaluate all proposals of the iteration at once, one thread per chain decides.
// Accepting flips buffer indices (model, tables, per-event sums); nothing is copied back
// and forth the way the reference backs up and restores its travel-time tables.
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/mcmceq_b200.h"
#include "chain.cuh"
#include "errors.h"
#include "forward.cuh"
#include "launch_count.h"
#include "sampler.cuh"
#include "state.h"
#include "tria.cuh"

namespace mq {

// ---- counter-based RNG ------------------------------------------------------------------
struct Philox {
    uint32_t key[2];
    uint32_t ctr[4];
    uint32_t out[4];
    uint64_t draws;   // number of 32-bit words consumed so far by this chain
    __device__ void block()
    {
        uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
#pragma unroll
        for (int r = 0; r < 10; r++) {
            const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
            c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
            k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
        }
        out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
    }
    __device__ Philox(uint64_t seed, uint32_t chain, uint64_t draws_)
    {
        key[0] = (uint32_t)seed; key[1] = (uint32_t)(seed >> 32);
        draws = draws_;
        ctr[2] = chain; ctr[3] = 0x6d636d63u;
        set_block(draws >> 2);
    }
    __device__ void set_block(uint64_t b) { ctr[0] = (uint32_t)b; ctr[1] = (uint32_t)(b >> 32); block(); }
    // 31 random bits, the range of libc rand()
    __device__ uint32_t next31()
    {
        const uint32_t w = out[draws & 3];
        draws++;
        if ((draws & 3) == 0) set_block(draws >> 2);
        return w >> 1;
    }
    // (float)rand()/RAND_MAX: uniform on [0,1], both ends possible (src/mcmc_eq.c:168-172)
    __device__ float uniform() { return (float)next31() / 2147483647.0f; }
    // rand_eq_int (src/mcmc_eq.c:162-166); the reference can return n when rand()==RAND_MAX, clamped here
    __device__ int below(int n)
    {
        const int i = (int)(uniform() * (float)n);
        return i < n ? i : n - 1;
    }
    // rand_eq_limited (src/mcmc_eq.c:174-178)
    __device__ float between(float lo, float hi) { return lo + (hi - lo) * (float)next31() / 2147483647.0f; }
    // rand_gauss: polar Box-Muller, second variate discarded (src/mcmc_eq.c:122-135)
    __device__ float gauss()
    {
        float v1, v2, s;
        do {
            v1 = 2.0f * uniform() - 1.f;
            v2 = 2.0f * uniform() - 1.f;
            s = v1 * v1 + v2 * v2;
        } while (s >= 1.0f);
        if (s == 0.0f) return 0.0f;
        return (float)((double)v1 * sqrt(-2.0 * log((double)s) / (double)s));
    }
    // rand_gauss_bounded (src/mcmc_eq.c:149-159): redraw until strictly inside (lo, hi).  The
    // reference loops for ever when that cannot happen; here the draw gives up (ok = false).
    __device__ float gauss_bounded(float v0, float sdev, float lo, float hi, bool* ok)
    {
        for (int tries = 0; tries < 100000; tries++) {
            const float dv = gauss() * sdev;
            if ((v0 + dv) > lo && (v0 + dv) < hi) return dv;
        }
        *ok = false;
        return 0.f;
    }
};

// ---- model_valid (src/mcmc_eq.c:180-229) on a model in global memory ---------------------
// Work arrays wz/wp/ws hold the depth-sorted copy.  Returns 0 when valid, 1 otherwise.
__device__ int model_valid_dev(int dim, const float* z, const float* vp, const float* vpvs, float* wz, float* wp,
                               float* ws, float dz, float zmin, float zmax, float inv_control)
{
    if (dim == 1) return 0;
    for (int i = 0; i < dim; i++) { wz[i] = z[i]; wp[i] = vp[i]; ws[i] = __fdiv_rn(vp[i], vpvs[i]); }
    // insertion sort == the reference's bubble sort (both stable, strict > comparisons)
    for (int i = 1; i < dim; i++) {
        const float kz = wz[i], kp = wp[i], ks = ws[i];
        int j = i - 1;
        while (j >= 0 && wz[j] > kz) { wz[j + 1] = wz[j]; wp[j + 1] = wp[j]; ws[j + 1] = ws[j]; j--; }
        wz[j + 1] = kz; wp[j + 1] = kp; ws[j + 1] = ks;
    }
    float thin = 3.402823466e+38f, prev = zmin;
    int lvz = 0;
    for (int i = 0; i < dim; i++) {
        const float bd = (i < dim - 1) ? (float)((double)__fadd_rn(wz[i], wz[i + 1]) / 2.0) : zmax;
        const float th = __fsub_rn(bd, prev);
        if (th < thin) thin = th;
        prev = bd;
        if (i < dim - 1) { if (wp[i] > wp[i + 1]) lvz++; if (ws[i] > ws[i + 1]) lvz++; }
    }
    if ((double)thin < sqrt((double)__fmul_rn(inv_control, inv_control)) * (double)dz) return 1;
    if (inv_control < 0.f && lvz > 0) return 1;
    return 0;
}

__device__ int find_in_cell_dev(const float* z, int dim, float zq)
{
    float best = 3.402823466e+38f;
    int k = 0;
    for (int i = 0; i < dim; i++) {
        const float d = __fsub_rn(z[i], zq), d2 = __fmul_rn(d, d);
        if (d2 <= best) { best = d2; k = i; }
    }
    return k;
}
__device__ int find_neighbor_dev(const float* z, int dim, int n)
{
    float best = 3.402823466e+38f;
    int k = 0;
    for (int i = 0; i < dim; i++) {
        if (i == n) continue;
        const float d = __fsub_rn(z[i], z[n]), d2 = __fmul_rn(d, d);
        if (d2 <= best) { best = d2; k = i; }
    }
    return k;
}

#define MQ_PI 3.141592653   // src/mc.h:50

// Chain c's current model (buffer mcur[c]) and the origin times of its current event buffer (ecur[c]).
struct CurModel {
    int mc, ec, dim;
    const float *z, *vp, *vpvs;
    const float* origin;   // [ne]
};
__device__ __forceinline__ CurModel cur_model(const Handle& hd, int c)
{
    CurModel m;
    m.mc = hd.mcur[c]; m.ec = hd.ecur[c];
    m.dim = hd.dim[m.mc * hd.n + c];
    const size_t mo = ((size_t)m.mc * hd.n + c) * hd.md;
    m.z = hd.z + mo; m.vp = hd.vp + mo; m.vpvs = hd.vpvs + mo;
    m.origin = hd.origin + ((size_t)m.ec * hd.n + c) * hd.ne;
    return m;
}

// The view of a chain before its proposal is known: nothing to evaluate, the current buffers.
__device__ __forceinline__ void view_defaults(const Handle& hd, const EvalView& v, int c, const CurModel& m)
{
    v.q_idx[c] = -1; v.r_idx[c] = -1; v.ev_only[c] = -2;
    v.mbuf[c] = m.mc; v.tbuf[2 * c] = hd.tcur[2 * c]; v.tbuf[2 * c + 1] = hd.tcur[2 * c + 1]; v.ebuf[c] = m.ec;
}

// A velocity-model proposal of `newdim` nuclei, written into the other model buffer: every event is evaluated with it into
// the other event buffer; calct (1 P, 2 S, 3 both) names the phases whose tables it needs.
__device__ __forceinline__ void view_model_arm(const Handle& hd, const SamplerDev& s, const EvalView& v, int c, const CurModel& m,
                                               int newdim, int calct)
{
    hd.dim[(1 - m.mc) * hd.n + c] = newdim;
    v.mbuf[c] = 1 - m.mc; v.ev_only[c] = -1; v.ebuf[c] = 1 - m.ec;
    s.rebuilt[c] = calct;
}

// ---- table rebuild queue: the phases in calct get the chain's other table buffer ...
__device__ __forceinline__ void flip_tables(const Handle& hd, const EvalView& v, int c, int calct)
{
    for (int ph = 0; ph < 2; ph++)
        if (calct & (1 << ph)) v.tbuf[2 * c + ph] = 1 - hd.tcur[2 * c + ph];
}
// ... and become work items of the eikonal launch.  The rebuilds of one chain sit next to each other in the work list: its
// P and S solves of one source depth grow their boxes alike (same interfaces), which is what the lanes of a warp should
// have in common.
__device__ __forceinline__ void queue_tables(const Handle& hd, const EvalView& v, int c, int calct)
{
    int item = atomicAdd(hd.n_items, (calct == 3) ? 2 : 1);
    for (int ph = 0; ph < 2; ph++) {
        if (!(calct & (1 << ph))) continue;
        if (item < 2 * hd.n) {                  // cannot fail (two items per chain at most); never write past the lists
            hd.item_chain[item] = c; hd.item_phase[item] = ph;
            hd.item_tab[item] = hd.tab + (((size_t)v.tbuf[2 * c + ph] * hd.n + c) * 2 + ph) * hd.tab_stride;
        }
        item++;
    }
}

// ---- start models (src/mcmc_eq.c:549-630) ---------------------------------------------------
__global__ void init_chains_kernel(Handle hd, SamplerDev s)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= hd.n) return;
    const mq_config& g = hd.cfg;
    Philox rng(hd.seed, (uint32_t)(hd.chain_offset + c), 0);
    bool ok = true;
    const float inv = (g.inv_control > 0.f) ? -g.inv_control : g.inv_control;
    s.inv_control[c] = inv;
    float* z = hd.z + (size_t)c * hd.md;     // buffer 0
    float* vp = hd.vp + (size_t)c * hd.md;
    float* vpvs = hd.vpvs + (size_t)c * hd.md;
    float* wz = s.wz + (size_t)c * hd.md; float* wp = s.wvp + (size_t)c * hd.md; float* ws = s.wvs + (size_t)c * hd.md;
    int dim = 1;
    for (int attempt = 0; attempt < 100000; attempt++) {
        if (g.start_cell_number > 1)
            dim = g.start_cell_number + (int)rng.gauss_bounded((float)g.start_cell_number, (float)g.sdev_start_cell_number,
                                                                1.0f, (float)hd.nz, &ok);
        else dim = 1;
        if (dim < 1) dim = 1;
        int first = 0;
        if (g.tria == 1) {   // two fixed nuclei at the top and the bottom of the model (src/mcmc_eq.c:577-588)
            dim += 2; first = 2;
            z[0] = hd.zmin; z[1] = hd.zmax;
            for (int i = 0; i < 2; i++) {
                const float value = g.start_vp + (z[i] - g.grid.z0) * g.start_vp_grad;
                vp[i] = value + rng.gauss_bounded(value, g.sdev_start_vp, g.vpmin, g.vpmax, &ok);
                vpvs[i] = g.start_vpvs + rng.gauss_bounded(g.start_vpvs, g.sdev_start_vpvs, g.vpvsmin, g.vpvsmax, &ok);
            }
        }
        if (dim > hd.md) dim = hd.md;
        for (int i = first; i < dim; i++) z[i] = rng.between(hd.zmin, hd.zmax);
        for (int i = first; i < dim; i++) {
            const float value = g.start_vp + (z[i] - g.grid.z0) * g.start_vp_grad;
            vp[i] = value + rng.gauss_bounded(value, g.sdev_start_vp, g.vpmin, g.vpmax, &ok);
            vpvs[i] = g.start_vpvs + rng.gauss_bounded(g.start_vpvs, g.sdev_start_vpvs, g.vpvsmin, g.vpvsmax, &ok);
        }
        if (model_valid_dev(dim, z, vp, vpvs, wz, wp, ws, g.grid.h, hd.zmin, hd.zmax, inv) == 0) break;
    }
    hd.dim[c] = dim;
    hd.mcur[c] = 0; hd.tcur[2 * c] = 0; hd.tcur[2 * c + 1] = 0; hd.ecur[c] = 0;
    float* eq = hd.eq + (size_t)c * hd.ne * 3;
    const float hx = (hd.xmax - hd.xmin) / 2.0f, hy = (hd.ymax - hd.ymin) / 2.0f;
    for (int q = 0; q < hd.ne; q++) eq[3 * q] = rng.between(hd.xmin + hx * (1.0f - g.r_start_eqh), hd.xmin + hx * (1.0f + g.r_start_eqh));
    for (int q = 0; q < hd.ne; q++) eq[3 * q + 1] = rng.between(hd.ymin + hy * (1.0f - g.r_start_eqh), hd.ymin + hy * (1.0f + g.r_start_eqh));
    for (int q = 0; q < hd.ne; q++) eq[3 * q + 2] = rng.between(hd.zmin, hd.zmax * g.r_start_eqv);
    for (int q = 0; q < hd.ne; q++)
        for (int k = 0; k < 3; k++)
            if (hd.pk.fix[3 * q + k] != -9999.0) eq[3 * q + k] = (float)hd.pk.fix[3 * q + k];
    float* pres = hd.pres + (size_t)c * hd.ns;
    float* sres = hd.sres + (size_t)c * hd.ns;
    for (int i = 0; i < hd.ns; i++) pres[i] = g.start_delay + rng.gauss_bounded(g.start_delay, g.sdev_start_delay, g.residual_min, g.residual_max, &ok);
    for (int i = 0; i < hd.ns; i++) sres[i] = g.start_delay + rng.gauss_bounded(g.start_delay, g.sdev_start_delay, g.residual_min, g.residual_max, &ok);
    if (g.scor_flag == 1 || g.scor_flag == 2) pres[g.reference_station] = g.ref_statcor_P;
    if (g.scor_flag == 2) sres[g.reference_station] = g.ref_statcor_S;
    for (int k = 0; k < 8; k++) hd.noise[8 * (size_t)c + k] = g.start_noise;
    s.draws[c] = rng.draws;
    s.acce[c] = 0; s.reject[c] = 0;
    for (int k = 0; k < 20; k++) s.counts[20 * (size_t)c + k] = 0;
    if (!ok) atomicOr(hd.err, kErrRetry);   // a start value could not be drawn inside its bounds (the reference would loop for ever)
}

// ---- proposal (src/mcmc_eq.c:856-1130) --------------------------------------------------------
__global__ void propose_kernel(Handle hd, SamplerDev s, EvalView v, int use_override)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= hd.n) return;
    const mq_config& g = hd.cfg;
    if (s.hold) {   // desynchronised stepping: parked chains keep their pending proposal, finished ones idle
        if (s.hold[c] == 2) { atomicAdd(&s.pass_stat[0], 1); return; }
        if (s.todo[c] <= 0) { s.hold[c] = 1; return; }
        s.hold[c] = 0;
    }
    const CurModel m = cur_model(hd, c);
    view_defaults(hd, v, c, m);
    s.kind[c] = 0; s.not_valid[c] = 0; s.rebuilt[c] = 0; s.log_fac[c] = 0.0;

    const long j = (long)s.acce[c];
    if (j >= (long)g.j_max_start + (long)g.j_max_main) return;   // chain finished (src/mcmc_eq.c:845)

    Philox rng(hd.seed, (uint32_t)(hd.chain_offset + c), s.draws[c]);
    float inv = s.inv_control[c];
    const int revert = (int)(g.j_max_start + g.j_max_main / 2);   // src/mcmc_eq.c:840
    if (j == revert && hd.lvz_flag == 1) { inv = -inv; s.inv_control[c] = inv; }   // fires every iteration while acce == revert (:849-853)

    char kind;
    float fac;
    if (use_override) { kind = s.ps_over[rng.below(s.len_over)]; fac = (j <= g.j_max_start) ? g.epi_search : 1.0f; }
    else if (j <= g.j_max_start) { kind = s.ps_start[rng.below(s.len_start)]; fac = g.epi_search; }
    else { kind = s.ps_main[rng.below(s.len_main)]; fac = 1.0f; }
    s.kind[c] = kind;

    const int dim = m.dim;
    const float *z = m.z, *vp = m.vp, *vpvs = m.vpvs;
    const size_t po = ((size_t)(1 - m.mc) * hd.n + c) * hd.md;   // the proposal's model buffer
    float* nz_ = hd.z + po;
    float* nvp = hd.vp + po;
    float* nvpvs = hd.vpvs + po;
    float* wz = s.wz + (size_t)c * hd.md; float* wp = s.wvp + (size_t)c * hd.md; float* ws = s.wvs + (size_t)c * hd.md;
    bool ok = true;
    int calct = 0, newdim = dim;
    bool model_arm = false;
    const int kMaxTries = 100000;

    switch (kind) {
    case 'Q': {
        const int idx = rng.below(hd.ne);
        const float* q = hd.eq + ((size_t)c * hd.ne + idx) * 3;
        float dx = rng.gauss_bounded(q[0], g.sdevxs * fac, hd.xmin, hd.xmax, &ok);
        float dy = rng.gauss_bounded(q[1], g.sdevys * fac, hd.ymin, hd.ymax, &ok);
        float dz = rng.gauss_bounded(q[2], g.sdevzs * fac, hd.zmin, hd.zmax, &ok);
        if (hd.pk.fix[3 * idx] != -9999.0) dx = 0.f;
        if (hd.pk.fix[3 * idx + 1] != -9999.0) dy = 0.f;
        if (hd.pk.fix[3 * idx + 2] != -9999.0) dz = 0.f;
        v.q_idx[c] = idx;
        v.q_xyz[3 * c] = q[0] + dx; v.q_xyz[3 * c + 1] = q[1] + dy; v.q_xyz[3 * c + 2] = q[2] + dz;
        v.ev_only[c] = idx;
        break;
    }
    case 'R': {
        const int idx = rng.below(hd.ns);
        float dx = rng.gauss_bounded(hd.pres[(size_t)c * hd.ns + idx], g.sdevresidual, g.residual_min, g.residual_max, &ok);
        float dy = rng.gauss_bounded(hd.sres[(size_t)c * hd.ns + idx], g.sdevresidual, g.residual_min, g.residual_max, &ok);
        if (g.scor_flag == -1) dy = 0.f;
        if (g.scor_flag == -2) dx = 0.f;
        float dx2 = 0.f, dy2 = 0.f;
        if (g.scor_flag != 0) {   // second addition of the reference (:919-928); for flags -1/-2 dx is applied twice
            dx2 = dx; dy2 = dy;
            if (g.reference_station == idx) {
                if (g.scor_flag == 1) dx2 = 0.f;
                if (g.scor_flag == 2) { dx2 = 0.f; dy2 = 0.f; }
            }
        }
        v.r_idx[c] = idx;
        v.r_d[4 * c] = dx; v.r_d[4 * c + 1] = dy; v.r_d[4 * c + 2] = dx2; v.r_d[4 * c + 3] = dy2;
        v.ev_only[c] = -1; v.ebuf[c] = 1 - m.ec;
        break;
    }
    case 'P': case 'V': case 'M': {
        // the two end nuclei of a linear-gradient model are never moved (src/mcmc_eq.c:990-998)
        const int fixed = (g.tria == 1) ? 2 : 0;
        if (kind == 'M' && !(dim > 1 + fixed)) { s.not_valid[c] = 1; break; }
        int t;
        for (t = 0; t < kMaxTries; t++) {
            for (int i = 0; i < dim; i++) { nz_[i] = z[i]; nvp[i] = vp[i]; nvpvs[i] = vpvs[i]; }
            const int idx = (kind == 'M') ? fixed + rng.below(dim - fixed) : rng.below(dim);
            if (kind == 'P') nvp[idx] = vp[idx] + rng.gauss_bounded(vp[idx], g.sdevvp, g.vpmin, g.vpmax, &ok);
            else if (kind == 'V') nvpvs[idx] = vpvs[idx] + rng.gauss_bounded(vpvs[idx], g.sdevvpvs, g.vpvsmin, g.vpvsmax, &ok);
            else nz_[idx] = z[idx] + rng.gauss_bounded(z[idx], g.sdevz, hd.zmin, hd.zmax, &ok);
            if (model_valid_dev(dim, nz_, nvp, nvpvs, wz, wp, ws, g.grid.h, hd.zmin, hd.zmax, inv) == 0) break;
        }
        if (t == kMaxTries) ok = false;
        calct = (kind == 'V') ? 2 : 3;
        model_arm = true;
        break;
    }
    case 'B': {
        if (!((double)(dim + 1) < ((double)g.max_dim / (1.0 + sqrt((double)(inv * inv))))) || dim + 1 > hd.md) { s.not_valid[c] = 1; break; }
        int t, idx = 0;
        for (t = 0; t < kMaxTries; t++) {
            for (int i = 0; i < dim; i++) { nz_[i] = z[i]; nvp[i] = vp[i]; nvpvs[i] = vpvs[i]; }
            const float newz = rng.between(hd.zmin, hd.zmax);
            idx = find_in_cell_dev(z, dim, newz);
            const float dvp = rng.gauss_bounded(vp[idx], g.sdevvp, g.vpmin, g.vpmax, &ok);
            const float dvs = rng.gauss_bounded(vpvs[idx], g.sdevvpvs, g.vpvsmin, g.vpvsmax, &ok);
            nvp[dim] = vp[idx] + dvp; nvpvs[dim] = vpvs[idx] + dvs; nz_[dim] = newz;
            if (model_valid_dev(dim + 1, nz_, nvp, nvpvs, wz, wp, ws, g.grid.h, hd.zmin, hd.zmax, inv) == 0) break;
        }
        if (t == kMaxTries) ok = false;
        newdim = dim + 1;
        {
            const float dv = nvp[dim] - nvp[idx], ds = nvpvs[dim] - nvpvs[idx];
            double lf = log((double)g.sdevvp * sqrt(2.0 * MQ_PI) / (double)(g.vpmax - g.vpmin)) +
                        (double)(dv * dv) / 2.0 / (double)g.sdevvp / (double)g.sdevvp;
            if (g.sdevvpvs != 0.f)
                lf = lf + log((double)g.sdevvpvs * sqrt(2.0 * MQ_PI) / (double)(g.vpvsmax - g.vpvsmin)) +
                     (double)(ds * ds) / 2.0 / (double)g.sdevvpvs / (double)g.sdevvpvs;
            s.log_fac[c] = lf;
        }
        calct = 3; model_arm = true;
        break;
    }
    case 'D': {
        const int fixed = (g.tria == 1) ? 2 : 0;   // ... nor removed (src/mcmc_eq.c:1059-1067)
        if (!(dim > 1 + fixed)) { s.not_valid[c] = 1; break; }
        int t;
        double lf = 0.0;
        for (t = 0; t < kMaxTries; t++) {
            const int dead = fixed + rng.below(dim - fixed);
            const int nb = find_neighbor_dev(z, dim, dead);
            const float dv = vp[dead] - vp[nb], ds = vpvs[dead] - vpvs[nb];
            lf = log((double)((g.vpmax - g.vpmin) / g.sdevvp) / sqrt(2.0 * MQ_PI)) -
                 (double)(dv * dv) / 2.0 / (double)g.sdevvp / (double)g.sdevvp;
            if (g.sdevvpvs != 0.f)
                lf = lf + log((double)((g.vpvsmax - g.vpvsmin) / g.sdevvpvs) / sqrt(2.0 * MQ_PI)) -
                     (double)(ds * ds) / 2.0 / (double)g.sdevvpvs / (double)g.sdevvpvs;
            for (int i = 0, k = 0; i < dim; i++) if (i != dead) { nz_[k] = z[i]; nvp[k] = vp[i]; nvpvs[k] = vpvs[i]; k++; }
            if (model_valid_dev(dim - 1, nz_, nvp, nvpvs, wz, wp, ws, g.grid.h, hd.zmin, hd.zmax, inv) == 0) break;
        }
        if (t == kMaxTries) ok = false;
        newdim = dim - 1;
        s.log_fac[c] = lf;
        calct = 3; model_arm = true;
        break;
    }
    case 'N': {
        const float* o = hd.noise + 8 * (size_t)c;
        float* nn = s.noise_new + 8 * (size_t)c;
        double lf = 0.0;
        // draw order p0,s0,p1,s1,... == index order 2*class+phase (:1097-1112)
        for (int k = 0; k < 8; k++) nn[k] = o[k] + rng.gauss_bounded(o[k], g.sdevn, g.noise_min, g.noise_max, &ok);
        for (int k = 0; k < 8; k++) lf = lf + (double)hd.n_class[k] * log((double)(o[k] / nn[k]));
        s.log_fac[c] = lf;
        v.ev_only[c] = -2;
        break;
    }
    default: s.not_valid[c] = 1; break;
    }

    if (model_arm) {
        view_model_arm(hd, s, v, c, m, newdim, calct);
        // a proposal whose retry loop gave up (!ok) is rejected without being evaluated: it queues no table rebuild
        if (g.eikonal == 1 && g.aflag != 1 && ok) {
            flip_tables(hd, v, c, calct);
            if (s.hold) s.hold[c] = 2;   // the tables are built later, together with those of other parked chains
            else queue_tables(hd, v, c, calct);
        }
    }
    if (g.aflag == 1) v.ev_only[c] = -2;   // prior sampling: no likelihood (src/misfit.c:61)
    if (!ok) { s.not_valid[c] = 2; v.ev_only[c] = -2; }   // a retry loop gave up: rejected whatever aflag (accept_kernel)
    s.draws[c] = rng.draws;
    if (s.hold) {
        if (s.hold[c] == 2) atomicAdd(&s.pass_stat[0], 1);
        else if (s.todo[c] > 1) atomicAdd(&s.pass_stat[1], 1);
    }
}

// Desynchronised stepping, the pass that builds tables: every parked chain queues its table rebuilds and is evaluated
// and decided in this pass, every other chain idles.
__global__ void flush_parked_kernel(Handle hd, SamplerDev s, EvalView v)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= hd.n) return;
    if (s.hold[c] != 2) {
        s.hold[c] = 1;
        if (s.todo[c] > 0) atomicAdd(&s.pass_stat[1], 1);
        return;
    }
    s.hold[c] = 0;
    queue_tables(hd, v, c, s.rebuilt[c]);   // propose_kernel chose the table buffers when the chain parked
    if (s.todo[c] > 1) atomicAdd(&s.pass_stat[1], 1);
}

// ---- replay: the proposal comes from a recorded stream instead of the RNG ------------------------------
// Fills exactly what propose_kernel fills, from injected data: s.kind[c] the arm, the proposed model in the work
// arrays s.wz/wvp/wvs (+ s.r_dim), the proposed event in v.q_xyz (+ s.r_qidx), the proposed station corrections in
// v.pres_over/sres_over, the proposed sigmas in s.noise_new, the proposal ratio in s.log_fac.  No validity test and no
// eligibility test: the recorded proposals passed the reference's own (src/mcmc_eq.c:945-951,1021,1059).
__global__ void replay_setup_kernel(Handle hd, SamplerDev s, EvalView v)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= hd.n) return;
    const CurModel m = cur_model(hd, c);
    view_defaults(hd, v, c, m);
    s.not_valid[c] = 0; s.rebuilt[c] = 0;
    const char kind = (char)s.kind[c];
    if (kind == 0) return;
    int calct = 0;
    switch (kind) {
    case 'Q': v.q_idx[c] = s.r_qidx[c]; v.ev_only[c] = s.r_qidx[c]; break;      // v.q_xyz was uploaded
    case 'R': v.r_idx[c] = -2; v.ev_only[c] = -1; v.ebuf[c] = 1 - m.ec; break;
    case 'N': v.ev_only[c] = -2; break;
    case 'V': calct = 2; break;
    case 'P': case 'M': case 'B': case 'D': calct = 3; break;
    default: s.not_valid[c] = 1; break;
    }
    if (calct) {
        const int d = s.r_dim[c];
        const size_t po = ((size_t)(1 - m.mc) * hd.n + c) * hd.md, wo = (size_t)c * hd.md;
        for (int i = 0; i < d; i++) { hd.z[po + i] = s.wz[wo + i]; hd.vp[po + i] = s.wvp[wo + i]; hd.vpvs[po + i] = s.wvs[wo + i]; }
        view_model_arm(hd, s, v, c, m, d, calct);
        if (hd.cfg.eikonal == 1 && hd.cfg.aflag != 1) {
            flip_tables(hd, v, c, calct);
            queue_tables(hd, v, c, calct);
        }
    }
    if (hd.cfg.aflag == 1) v.ev_only[c] = -2;
}

// ---- accept / reject (src/mcmc_eq.c:1135-1191) -------------------------------------------------
__global__ void accept_kernel(Handle hd, SamplerDev s, EvalView v)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= hd.n) return;
    if (s.hold) {   // desynchronised stepping: only chains evaluated in this pass are decided; an iteration is used up
        if (s.hold[c] != 0) return;
        s.todo[c]--;
    }
    const char kind = (char)s.kind[c];
    if (kind == 0) return;   // finished chain
    const mq_config& g = hd.cfg;
    const int n = hd.n;
    int64_t* cnt = s.counts + 20 * (size_t)c;
    const int slot = (kind == 'N') ? 0 : (kind == 'P') ? 1 : (kind == 'V') ? 2 : (kind == 'Q') ? 3 : (kind == 'R') ? 4
                   : (kind == 'M') ? 5 : (kind == 'B') ? 6 : 7;
    const int not_valid = s.not_valid[c];
    float mf[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const float* noise = (kind == 'N') ? s.noise_new + 8 * (size_t)c : hd.noise + 8 * (size_t)c;
    float alpha;
    double new_misfit = 0, new_rms = 0, new_ll = 0;
    if (not_valid) {
        alpha = 0.f;   // ineligible move (1) or a retry loop that gave up (2): still consumes a uniform (quirk Q5)
    } else {
        for (int k = 0; k < 8; k++) mf[k] = (g.aflag == 1) ? 0.f : hd.mf_eval[8 * (size_t)c + k];
        new_misfit = chain_misfit(mf, noise);
        new_rms = chain_rms(mf, hd.sum_of_picks);
        new_ll = -new_misfit / 2.0;
        // parallel tempering (comm.cu): the likelihood enters with the chain's inverse temperature; for the noise arm
        // log_fac is the likelihood's normalisation term (src/mcmc_eq.c:1114-1117) and is tempered with it.  beta == 1
        // (the default, and the reference) leaves every operand unchanged.
        const double beta = hd.beta ? (double)hd.beta[c] : 1.0;
        alpha = chain_alpha((kind == 'N') ? beta * s.log_fac[c] : s.log_fac[c], beta * new_ll, beta * hd.ll[c]);
        cnt[0]++;   // nmod: models whose misfit was evaluated
    }
    if (g.aflag == 1) alpha = 1.f;
    if (not_valid && g.aflag == 0) alpha = 0.f;
    // a retry loop that gave up leaves its last rejected try in the proposal buffers: never installed, not even when
    // sampling the prior (the reference would loop for ever there)
    if (not_valid == 2) alpha = 0.f;

    float u;
    if (s.u_inject) u = s.u_inject[c];   // replay: the reference's own deviate, no draw is consumed
    else {
        Philox rng(hd.seed, (uint32_t)(hd.chain_offset + c), s.draws[c]);
        u = rng.uniform();
        s.draws[c] = rng.draws;
    }
    if (s.r_alpha) { s.r_alpha[c] = alpha; s.r_accept[c] = (u < alpha) ? 1 : 0; s.r_newll[c] = new_ll; }

    if (u < alpha) {
        const int64_t number = s.acce[c];
        s.acce[c] = number + 1;
        cnt[1 + 2 * slot]++;
        cnt[17]++;
        // apply the proposal
        if (kind == 'Q') {
            const int idx = v.q_idx[c];
            float* q = hd.eq + ((size_t)c * hd.ne + idx) * 3;
            q[0] = v.q_xyz[3 * c]; q[1] = v.q_xyz[3 * c + 1]; q[2] = v.q_xyz[3 * c + 2];
            if (g.aflag != 1) {
                const int ec = hd.ecur[c];
                float* es = hd.evsum + (((size_t)ec * n + c) * hd.ne + idx) * 8;
                for (int k = 0; k < 8; k++) es[k] = hd.evq[8 * (size_t)c + k];
                hd.origin[((size_t)ec * n + c) * hd.ne + idx] = hd.oq[c];
            }
        } else if (kind == 'R') {
            const int idx = v.r_idx[c];
            const float dx = v.r_d[4 * c], dy = v.r_d[4 * c + 1], dx2 = v.r_d[4 * c + 2], dy2 = v.r_d[4 * c + 3];
            float* pres = hd.pres + (size_t)c * hd.ns;
            float* sres = hd.sres + (size_t)c * hd.ns;
            const float nsm1 = (float)(hd.ns - 1);
            if (idx == -2) {   // replay: the proposed corrections were given in full
                for (int k = 0; k < hd.ns; k++) { pres[k] = v.pres_over[(size_t)c * hd.ns + k]; sres[k] = v.sres_over[(size_t)c * hd.ns + k]; }
            } else if (g.scor_flag <= 0)
                for (int k = 0; k < hd.ns; k++) {
                    pres[k] = (k == idx) ? __fadd_rn(pres[k], dx) : __fsub_rn(pres[k], __fdiv_rn(dx, nsm1));
                    sres[k] = (k == idx) ? __fadd_rn(sres[k], dy) : __fsub_rn(sres[k], __fdiv_rn(dy, nsm1));
                }
            if (idx != -2 && g.scor_flag != 0) { pres[idx] = __fadd_rn(pres[idx], dx2); sres[idx] = __fadd_rn(sres[idx], dy2); }
            if (g.aflag != 1) hd.ecur[c] = v.ebuf[c];
        } else if (kind == 'N') {
            for (int k = 0; k < 8; k++) hd.noise[8 * (size_t)c + k] = noise[k];
        } else {   // P V M B D
            hd.mcur[c] = v.mbuf[c];
            hd.tcur[2 * c] = v.tbuf[2 * c];
            hd.tcur[2 * c + 1] = v.tbuf[2 * c + 1];
            if (g.aflag != 1) hd.ecur[c] = v.ebuf[c];
        }
        {
            for (int k = 0; k < 8; k++) hd.mf[8 * (size_t)c + k] = mf[k];
            hd.ll[c] = new_ll; hd.rms[c] = new_rms; hd.misfit[c] = new_misfit;
        }
        // decimated output (src/mcmc_eq.c:1163) and best model (src/mcmc_eq.c:1186-1191)
        const int64_t acce = number + 1;
        if (g.deci > 0 && (acce / g.deci) * g.deci == acce) {
            const int pending = s.ring.wr[c] - *(volatile int32_t*)&s.ring.rd[c];
            if (pending >= s.ring.slots) { s.ring.pend[c] = 2; s.ring.lost[c]++; }   // ring full: the record is dropped and counted
            else s.ring.pend[c] = 1;
            s.ring.number[c] = number; s.ring.code[c] = kind; s.ring.rms[c] = new_rms;
        }
        if (new_rms < s.best_rms[c]) { s.best_rms[c] = new_rms; s.best.flag[c] = 2; s.best.number[c] = number; s.best.rms[c] = new_rms; }
    } else {
        s.reject[c]++;
        cnt[2 + 2 * slot]++;
        cnt[18]++;
    }
}

// ---- snapshots: one block per chain copies the current state when asked to ----------------------
__device__ void snapshot_copy(const Handle& hd, const Snapshot& d, int c)
{
    const CurModel m = cur_model(hd, c);
    const int md = hd.md, ne = hd.ne, ns = hd.ns;
    for (int i = threadIdx.x; i < m.dim; i += blockDim.x) {
        d.z[(size_t)c * md + i] = m.z[i]; d.vp[(size_t)c * md + i] = m.vp[i]; d.vpvs[(size_t)c * md + i] = m.vpvs[i];
    }
    for (int i = threadIdx.x; i < 3 * ne; i += blockDim.x) d.eq[(size_t)c * ne * 3 + i] = hd.eq[(size_t)c * ne * 3 + i];
    for (int i = threadIdx.x; i < ne; i += blockDim.x) d.origin[(size_t)c * ne + i] = m.origin[i];
    for (int i = threadIdx.x; i < ns; i += blockDim.x) { d.pres[(size_t)c * ns + i] = hd.pres[(size_t)c * ns + i]; d.sres[(size_t)c * ns + i] = hd.sres[(size_t)c * ns + i]; }
    if (threadIdx.x < 8) d.noise[8 * (size_t)c + threadIdx.x] = hd.noise[8 * (size_t)c + threadIdx.x];
    if (threadIdx.x == 0) d.dim[c] = m.dim;
}

// The chain's current state as one packed record (layout: struct Ring).
__device__ void record_write(const Handle& hd, const Ring& R, int c, float* rec)
{
    const CurModel m = cur_model(hd, c);
    const int md = hd.md, ne = hd.ne, ns = hd.ns;
    if (threadIdx.x == 0) {
        int32_t* hi = (int32_t*)rec;
        hi[0] = c; hi[1] = R.code[c]; hi[2] = m.dim; hi[3] = 0;
        *(int64_t*)(rec + 4) = R.number[c];
        *(double*)(rec + 6) = R.rms[c];
    }
    float* o = rec + kRecHead;
    if (threadIdx.x < 8) o[threadIdx.x] = hd.noise[8 * (size_t)c + threadIdx.x];
    o += 8;
    for (int i = threadIdx.x; i < m.dim; i += blockDim.x) { o[i] = m.z[i]; o[md + i] = m.vp[i]; o[2 * md + i] = m.vpvs[i]; }
    o += 3 * md;
    for (int i = threadIdx.x; i < 3 * ne; i += blockDim.x) o[i] = hd.eq[(size_t)c * ne * 3 + i];
    o += 3 * ne;
    for (int i = threadIdx.x; i < ne; i += blockDim.x) o[i] = m.origin[i];
    o += ne;
    for (int i = threadIdx.x; i < ns; i += blockDim.x) { o[i] = hd.pres[(size_t)c * ns + i]; o[ns + i] = hd.sres[(size_t)c * ns + i]; }
}

// Drain, device side (copy stream): the published records [rd, wr) of every chain move to the staging buffer, one
// chain's records next to each other in order; count[0] = records packed, count[1] = records dropped since the last drain.
__global__ void __launch_bounds__(128) pack_records_kernel(int n, Ring R, float* stage, int cap_records, int32_t* count)
{
    const int c = blockIdx.x;
    __shared__ int base;
    const int w = *(volatile int32_t*)&R.wr[c], r = R.rd[c];
    int k = w - r;
    __threadfence();
    if (threadIdx.x == 0) {
        const int l = atomicExch(&R.lost[c], 0);
        if (l) atomicAdd(&count[1], l);
        base = 0;
        if (k > 0) {
            base = atomicAdd(&count[0], k);
            if (base + k > cap_records) { atomicSub(&count[0], k); base = -1; }   // staging full: the records stay in the ring
        }
    }
    __syncthreads();
    if (k <= 0 || base < 0) return;
    const int nv = R.rec_floats / 4;
    for (int j = 0; j < k; j++) {
        const float4* src = (const float4*)(R.data + ((size_t)c * R.slots + (r + j) % R.slots) * R.rec_floats);
        float4* dst = (float4*)(stage + (size_t)(base + j) * R.rec_floats);
        for (int i = threadIdx.x; i < nv; i += blockDim.x) dst[i] = src[i];
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) *(volatile int32_t*)&R.rd[c] = w;
}

// Vp and Vp/Vs of a model at depth node i as analyse_eq bins them (src/analyse_eq.c:564-606): the nearest nucleus, or with
// TRIA = 1 the interpolated profile (:573-580,593-598), clipped to the prior range.  *nearest: the nucleus taken (-1 with
// TRIA = 1).  The posterior and the diagnostics both rasterise through here.
__device__ void node_velocity(const mq_config& g, const float* z, const float* vp, const float* vpvs, int dim, int i, float* vv_out,
                              float* rr_out, int* nearest)
{
    const float zz = __fadd_rn(__fmul_rn((float)i, g.grid.h), g.grid.z0);
    float vv, rr;
    if (g.tria == 1) {
        int lo, hi;
        tria::segment_of_node(z, dim, i, g.grid.h, g.grid.z0, &lo, &hi);
        vv = tria::line_through(zz, z[lo], vp[lo], z[hi], vp[hi]);
        rr = tria::line_through(zz, z[lo], vpvs[lo], z[hi], vpvs[hi]);
        *nearest = -1;
    } else {
        const int k = find_in_cell_dev(z, dim, zz);
        vv = vp[k];
        rr = vpvs[k];
        *nearest = k;
    }
    if (vv > g.vpmax) vv = g.vpmax;
    if (vv < g.vpmin) vv = g.vpmin;
    if (rr > g.vpvsmax) rr = g.vpvsmax;
    if (rr < g.vpvsmin) rr = g.vpvsmin;
    *vv_out = vv;
    *rr_out = rr;
}

// analyse_eq pass 1 for one decimated model (src/analyse_eq.c:564-640): per depth node the velocity of the nearest
// nucleus, clipped to the prior range, goes into the Vp and Vp/Vs histograms; hypocentres, origin times, station
// corrections and sigmas into running sums.
__device__ void posterior_accumulate(const Handle& hd, int c)
{
    const Posterior& P = hd.post;
    const CurModel m = cur_model(hd, c);
    const int dim = m.dim, nz = hd.nz, ne = hd.ne, ns = hd.ns;
    const float *z = m.z, *vp = m.vp, *vpvs = m.vpvs;
    int32_t* hist_vp = P.iblock;
    int32_t* hist_vs = hist_vp + (size_t)P.ndv * nz;
    int32_t* boundary = hist_vs + (size_t)P.ndvpvs * nz;
    double* vsum = P.dblock;
    double* eqsum = vsum + 4 * (size_t)nz;
    double* ressum = eqsum + 8 * (size_t)ne;
    double* noisesum = ressum + 4 * (size_t)ns;
    const mq_config& g = hd.cfg;
    for (int i = threadIdx.x; i < nz; i += blockDim.x) {
        float vv, rr;
        int k;
        node_velocity(g, z, vp, vpvs, dim, i, &vv, &rr, &k);
        if (k >= 0) {   // a layer boundary at node i: the nucleus above is another one (no boundaries with TRIA = 1)
            const float zz = __fadd_rn(__fmul_rn((float)i, g.grid.h), g.grid.z0);
            if (vp[k] != vp[find_in_cell_dev(z, dim, __fsub_rn(zz, g.grid.h))]) atomicAdd(&boundary[i], 1);
        }
        int j = (int)__fdiv_rn(__fsub_rn(vv, g.vpmin), P.dv);
        if (j > P.ndv - 1) j = P.ndv - 1;
        atomicAdd(&hist_vp[(size_t)j * nz + i], 1);
        j = (int)__fdiv_rn(__fsub_rn(rr, g.vpvsmin), P.dvpvs);
        if (j > P.ndvpvs - 1) j = P.ndvpvs - 1;
        atomicAdd(&hist_vs[(size_t)j * nz + i], 1);
        atomicAdd(&vsum[4 * i], (double)vv); atomicAdd(&vsum[4 * i + 1], (double)vv * vv);
        atomicAdd(&vsum[4 * i + 2], (double)rr); atomicAdd(&vsum[4 * i + 3], (double)rr * rr);
    }
    for (int e = threadIdx.x; e < ne; e += blockDim.x) {
        const float* q = hd.eq + ((size_t)c * ne + e) * 3;
        const double v[4] = {q[0], q[1], q[2], m.origin[e]};
        for (int k = 0; k < 4; k++) { atomicAdd(&eqsum[8 * e + k], v[k]); atomicAdd(&eqsum[8 * e + 4 + k], v[k] * v[k]); }
    }
    for (int i = threadIdx.x; i < ns; i += blockDim.x) {
        const double a = hd.pres[(size_t)c * ns + i], b = hd.sres[(size_t)c * ns + i];
        atomicAdd(&ressum[4 * i], a); atomicAdd(&ressum[4 * i + 1], b);
        atomicAdd(&ressum[4 * i + 2], a * a); atomicAdd(&ressum[4 * i + 3], b * b);
    }
    if (threadIdx.x < 8) {
        const double v = hd.noise[8 * (size_t)c + threadIdx.x];
        atomicAdd(&noisesum[threadIdx.x], v); atomicAdd(&noisesum[8 + threadIdx.x], v * v);
    }
    if (threadIdx.x == 0) atomicAdd(&noisesum[16], 1.0);
}

// Convergence diagnostics for one used model (DESIGN.md section 4d): quantity q of the record (q = 0 rms, 1 dim, 2..9 the
// sigmas, then Vp and Vp/Vs per depth node, x y z t per event, P and S correction per station) goes into the chain's open
// batch slot as d = x - ref.  Threads over quantities; each (chain, quantity) is summed in the same order whatever the
// stepping, so the accumulators are a function of the chain's records alone.
__device__ void diag_accumulate(const Handle& hd, const Ring& R, int c)
{
    const Diag& D = hd.diag;
    const CurModel cm = cur_model(hd, c);
    const int Q = D.Q, K = D.K, nz = hd.nz, ne = hd.ne;
    const int64_t m = D.n_models[c];
    const int k = D.full_batches[c], L = D.batch_len[c];
    const bool fills = m + 1 - (int64_t)k * L == L;          // this model fills the open slot
    double* ref = D.ref + (size_t)c * Q;
    double* S = D.sum + (size_t)c * K * Q;
    double* T = D.sumsq + (size_t)c * K * Q;
    for (int q = threadIdx.x; q < Q; q += blockDim.x) {
        double x;
        if (q == 0) x = R.rms[c];
        else if (q == 1) x = (double)cm.dim;
        else if (q < 10) x = (double)hd.noise[8 * (size_t)c + q - 2];
        else if (q < 10 + 2 * nz) {
            const int i = (q - 10) % nz;
            float vv, rr;
            int near;
            node_velocity(hd.cfg, cm.z, cm.vp, cm.vpvs, cm.dim, i, &vv, &rr, &near);
            x = (double)(q < 10 + nz ? vv : rr);
        } else if (q < 10 + 2 * nz + 4 * ne) {
            const int e = (q - 10 - 2 * nz) >> 2, j = (q - 10 - 2 * nz) & 3;
            x = (double)(j < 3 ? hd.eq[((size_t)c * ne + e) * 3 + j] : cm.origin[e]);
        } else {
            const int st = (q - 10 - 2 * nz - 4 * ne) >> 1;
            x = (double)((q & 1) == 0 ? hd.pres[(size_t)c * hd.ns + st] : hd.sres[(size_t)c * hd.ns + st]);
        }
        if (m == 0) ref[q] = x;
        const double d = __dsub_rn(x, ref[q]);
        S[(size_t)k * Q + q] = __dadd_rn(S[(size_t)k * Q + q], d);
        T[(size_t)k * Q + q] = __dadd_rn(T[(size_t)k * Q + q], __dmul_rn(d, d));
        if (fills && k + 1 == K) {   // every slot full: pairs merge, slots K/2 .. K-1 are empty again
            for (int i = 0; i < K / 2; i++) {
                S[(size_t)i * Q + q] = __dadd_rn(S[(size_t)(2 * i) * Q + q], S[(size_t)(2 * i + 1) * Q + q]);
                T[(size_t)i * Q + q] = __dadd_rn(T[(size_t)(2 * i) * Q + q], T[(size_t)(2 * i + 1) * Q + q]);
            }
            for (int i = K / 2; i < K; i++) { S[(size_t)i * Q + q] = 0.0; T[(size_t)i * Q + q] = 0.0; }
        }
    }
    __syncthreads();   // every thread has read m, k and L
    if (threadIdx.x == 0) {
        D.n_models[c] = m + 1;
        if (fills) {
            if (k + 1 == K) { D.full_batches[c] = K / 2; D.batch_len[c] = 2 * L; }
            else D.full_batches[c] = k + 1;
        }
    }
}

// Hypocentre uncertainty for one used model (DESIGN.md section 4e): per event, v = (x, y, z, t) goes into the chain's
// sums of d = v - ref and of the ten products d_i d_j, and x, y, z into the event's histograms.  Threads over events; each
// (chain, event) is summed in record order whatever the stepping, and integer atomics give the same counts in any order.
__device__ void hypo_accumulate(const Handle& hd, int c)
{
    const Hypo& H = hd.hypo;
    const CurModel cm = cur_model(hd, c);
    const int ne = hd.ne, nbt = H.nb[0] + H.nb[1] + H.nb[2];
    const int64_t m = H.n_models[c];
    const float lo[3] = {hd.xmin, hd.ymin, hd.zmin}, hi[3] = {hd.xmax, hd.ymax, hd.zmax};
    double* ref = H.ref + (size_t)c * 4 * ne;
    double* S = H.sum + (size_t)c * 4 * ne;
    double* C = H.cross + (size_t)c * 10 * ne;
    for (int e = threadIdx.x; e < ne; e += blockDim.x) {
        const float* q = hd.eq + ((size_t)c * ne + e) * 3;
        const float v[4] = {q[0], q[1], q[2], cm.origin[e]};
        double d[4];
        for (int k = 0; k < 4; k++) {
            if (m == 0) ref[(size_t)k * ne + e] = (double)v[k];
            d[k] = __dsub_rn((double)v[k], ref[(size_t)k * ne + e]);
            S[(size_t)k * ne + e] = __dadd_rn(S[(size_t)k * ne + e], d[k]);
        }
        int p = 0;
        for (int i = 0; i < 4; i++)
            for (int j = i; j < 4; j++, p++) C[(size_t)p * ne + e] = __dadd_rn(C[(size_t)p * ne + e], __dmul_rn(d[i], d[j]));
        int32_t* row = H.hist + (size_t)e * nbt;
        for (int a = 0; a < 3; a++) {
            int j = (int)__fdiv_rn(__fsub_rn(v[a], lo[a]), H.bin);
            j = min(max(j, 0), H.nb[a] - 1);
            if (!(v[a] >= lo[a] && v[a] <= hi[a])) atomicAdd(&H.outside[3 * e + a], 1);
            atomicAdd(&row[j], 1);
            row += H.nb[a];
        }
    }
    __syncthreads();   // every thread has read m
    if (threadIdx.x == 0) H.n_models[c] = m + 1;
}

__global__ void snapshot_kernel(Handle hd, SamplerDev s)
{
    const int c = blockIdx.x;
    const int pend = s.ring.pend[c];
    if (pend) {
        if (hd.post.on && (long long)s.ring.number[c] > hd.post.burn_in) posterior_accumulate(hd, c);
        if (hd.diag.on && (long long)s.ring.number[c] > hd.diag.burn_in) diag_accumulate(hd, s.ring, c);
        if (hd.hypo.on && (long long)s.ring.number[c] > hd.hypo.burn_in) hypo_accumulate(hd, c);
        if (pend == 1) {
            const int wr = s.ring.wr[c];
            record_write(hd, s.ring, c, s.ring.data + ((size_t)c * s.ring.slots + wr % s.ring.slots) * s.ring.rec_floats);
            __threadfence();
            __syncthreads();
            if (threadIdx.x == 0) *(volatile int32_t*)&s.ring.wr[c] = wr + 1;   // published: a drain may take it
        }
        __syncthreads();
        if (threadIdx.x == 0) s.ring.pend[c] = 0;
    }
    if (s.best.flag[c] >= 2) {
        snapshot_copy(hd, s.best, c);
        __syncthreads();
        if (threadIdx.x == 0) s.best.flag[c] = 1;
    }
}

__global__ void init_best_kernel(int n, const double* rms, SamplerDev s)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    s.best_rms[c] = rms[c];
    s.best.flag[c] = 2; s.best.number[c] = 0; s.best.rms[c] = rms[c];
    s.ring.wr[c] = 0; s.ring.rd[c] = 0; s.ring.lost[c] = 0; s.ring.pend[c] = 0;
}

// ---- host side ---------------------------------------------------------------------------------
template <class T>
static cudaError_t dz(T** p, size_t count)
{
    cudaError_t e = cudaMalloc((void**)p, (count ? count : 1) * sizeof(T));
    if (e == cudaSuccess) e = cudaMemset(*p, 0, (count ? count : 1) * sizeof(T));
    return e;
}

static cudaError_t alloc_snapshot(Snapshot* d, const Handle* h)
{
    const size_t n = h->n;
    cudaError_t e;
    if ((e = dz(&d->dim, n))) return e;
    if ((e = dz(&d->z, n * h->md))) return e;
    if ((e = dz(&d->vp, n * h->md))) return e;
    if ((e = dz(&d->vpvs, n * h->md))) return e;
    if ((e = dz(&d->eq, n * h->ne * 3))) return e;
    if ((e = dz(&d->origin, n * h->ne))) return e;
    if ((e = dz(&d->pres, n * h->ns))) return e;
    if ((e = dz(&d->sres, n * h->ns))) return e;
    if ((e = dz(&d->noise, n * 8))) return e;
    if ((e = dz(&d->rms, n))) return e;
    if ((e = dz(&d->number, n))) return e;
    if ((e = dz(&d->code, n))) return e;
    if ((e = dz(&d->flag, n))) return e;
    return cudaSuccess;
}
static void free_snapshot(Snapshot* d)
{
    cudaFree(d->dim); cudaFree(d->z); cudaFree(d->vp); cudaFree(d->vpvs); cudaFree(d->eq); cudaFree(d->origin);
    cudaFree(d->pres); cudaFree(d->sres); cudaFree(d->noise); cudaFree(d->rms); cudaFree(d->number); cudaFree(d->code); cudaFree(d->flag);
}

// Balanced proposal strings (src/mcmc_eq.c:769-834): Q and R are repeated once per `per` events / stations.
static std::string balance(const char* letters, int noq, int nos, int per)
{
    std::string out;
    for (const char* q = letters; *q; q++) {
        switch (*q) {
        case 'Q': for (int j = 0; j < noq; j += per) out += 'Q'; break;
        case 'R': for (int j = 0; j < nos; j += per) out += 'R'; break;
        case 'N': case 'M': case 'V': case 'P': case 'B': case 'D': out += *q; break;
        default: break;
        }
    }
    return out;
}

static cudaError_t upload_string(char** d, const std::string& s)
{
    cudaFree(*d);
    *d = nullptr;
    cudaError_t e = cudaMalloc((void**)d, s.size() + 1);
    if (e == cudaSuccess) e = cudaMemcpy(*d, s.c_str(), s.size() + 1, cudaMemcpyHostToDevice);
    return e;
}

int sampler_get(Handle* h, Sampler** out)
{
    if (h->sampler) { *out = (Sampler*)h->sampler; return MQ_OK; }
    Sampler* s = new Sampler();
    memset((void*)static_cast<SamplerDev*>(s), 0, sizeof(SamplerDev));
    s->started = false;
    const size_t n = h->n;
#define TRY(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { set_error("%s: %s", #x, cudaGetErrorString(e_)); return MQ_ERR_CUDA; } } while (0)
    TRY(dz(&s->acce, n)); TRY(dz(&s->reject, n)); TRY(dz(&s->counts, n * 20)); TRY(dz(&s->draws, n));
    TRY(dz(&s->inv_control, n)); TRY(dz(&s->kind, n)); TRY(dz(&s->not_valid, n)); TRY(dz(&s->rebuilt, n));
    TRY(dz(&s->log_fac, n)); TRY(dz(&s->noise_new, n * 8)); TRY(dz(&s->best_rms, n));
    TRY(dz(&s->wz, n * h->md)); TRY(dz(&s->wvp, n * h->md)); TRY(dz(&s->wvs, n * h->md));
    TRY(alloc_snapshot(&s->best, h));
    {
        const char* e = getenv("MCMCEQ_RING_SLOTS");
        int slots = h->ring_slots > 0 ? h->ring_slots : (e ? atoi(e) : 4);
        if (slots < 1) slots = 1;
        if (slots > 64) slots = 64;
        s->ring.slots = slots;
        s->ring.rec_floats = rec_floats_of(h->md, h->ne, h->ns);
        TRY(dz(&s->ring.data, n * slots * s->ring.rec_floats));
        TRY(dz(&s->ring.wr, n)); TRY(dz(&s->ring.rd, n)); TRY(dz(&s->ring.lost, n)); TRY(dz(&s->ring.pend, n));
        TRY(dz(&s->ring.number, n)); TRY(dz(&s->ring.code, n)); TRY(dz(&s->ring.rms, n));
        TRY(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
        TRY(cudaEventCreateWithFlags(&s->ev_main, cudaEventDisableTiming));
        memset(s->batch, 0, sizeof s->batch);
    }
    TRY(dz(&s->u_buf, n)); TRY(dz(&s->r_alpha, n)); TRY(dz(&s->r_accept, n)); TRY(dz(&s->r_newll, n)); TRY(dz(&s->r_qidx, n));
    TRY(dz(&s->r_dim, n));
    TRY(dz(&s->todo_buf, n)); TRY(dz(&s->hold_buf, n)); TRY(dz(&s->stat_buf, 2));
    const std::string a = balance(h->cfg.dstring_start, h->ne, h->ns, 10), b = balance(h->cfg.dstring_main, h->ne, h->ns, 20);
    s->len_start = (int)a.size(); s->len_main = (int)b.size();
    TRY(upload_string(&s->ps_start, a)); TRY(upload_string(&s->ps_main, b));
    {
        std::vector<float> inv(n, h->inv_control);
        TRY(cudaMemcpy(s->inv_control, inv.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    }
#undef TRY
    h->sampler = s;
    *out = s;
    return MQ_OK;
}

void sampler_destroy(Handle* h)
{
    Sampler* s = (Sampler*)h->sampler;
    if (!s) return;
    cudaFree(s->acce); cudaFree(s->reject); cudaFree(s->counts); cudaFree(s->draws); cudaFree(s->inv_control);
    cudaFree(s->kind); cudaFree(s->not_valid); cudaFree(s->rebuilt); cudaFree(s->log_fac); cudaFree(s->noise_new);
    cudaFree(s->best_rms); cudaFree(s->wz); cudaFree(s->wvp); cudaFree(s->wvs);
    free_snapshot(&s->best);
    if (s->cur.dim) free_snapshot(&s->cur);
    if (s->copy_stream) cudaStreamSynchronize(s->copy_stream);
    cudaFree(s->ring.data); cudaFree(s->ring.wr); cudaFree(s->ring.rd); cudaFree(s->ring.lost); cudaFree(s->ring.pend);
    cudaFree(s->ring.number); cudaFree(s->ring.code); cudaFree(s->ring.rms);
    for (int i = 0; i < 2; i++) {
        mq_batch& b = s->batch[i];
        cudaFree(b.d_stage); cudaFree(b.d_count);
        if (b.h_count) cudaFreeHost(b.h_count);
        if (b.h_stage) cudaFreeHost(b.h_stage);
        if (b.ev_count) cudaEventDestroy(b.ev_count);
        if (b.ev_data) cudaEventDestroy(b.ev_data);
        delete b.order;
    }
    if (s->ev_main) cudaEventDestroy(s->ev_main);
    if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
    cudaFree(s->ps_start); cudaFree(s->ps_main); cudaFree(s->ps_over);
    cudaFree(s->u_buf); cudaFree(s->r_alpha); cudaFree(s->r_accept); cudaFree(s->r_newll); cudaFree(s->r_qidx); cudaFree(s->r_dim);
    cudaFree(s->todo_buf); cudaFree(s->hold_buf); cudaFree(s->stat_buf);
    cudaFree(h->prop_view.pres_over); cudaFree(h->prop_view.sres_over);
    h->prop_view.pres_over = nullptr; h->prop_view.sres_over = nullptr;
    delete s;
    h->sampler = nullptr;
}

}  // namespace mq

using namespace mq;

static int start_sampler_state(Handle* h, Sampler* s)
{
    // first forward of the start models and the "best so far" bookkeeping (src/mcmc_eq.c:739-765)
    int rc = forward_current_device(h, 3);
    if (rc != MQ_OK) return rc;
    init_best_kernel<<<(h->n + 127) / 128, 128, 0, h->stream>>>(h->n, h->rms, s->dev());
    count_launch();
    MQ_CUDA(cudaGetLastError());
    snapshot_kernel<<<h->n, 128, 0, h->stream>>>(*h, s->dev());
    count_launch();
    MQ_CUDA(cudaGetLastError());
    s->started = true;
    return check_device_errors(h);   // synchronises: solver status, invalid station correction, start values out of bounds
}

// The handle's sampler, its chains scored once before their first step (chains supplied through mq_set_models included).
static int started_sampler(Handle* h, Sampler** out)
{
    int rc = sampler_get(h, out);
    if (rc == MQ_OK && (!(*out)->started || !h->forward_done)) rc = start_sampler_state(h, *out);
    return rc;
}

extern "C" int mq_init_chains(mq_handle* hh)
{
    if (!hh) { set_error("mq_init_chains: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    MQ_CUDA(cudaSetDevice(h->device));
    Sampler* s;
    int rc = sampler_get(h, &s);
    if (rc != MQ_OK) return rc;
    if (s->len_start < 1 || s->len_main < 1) { set_error("mq_init_chains: empty proposal string (config line 33)"); return MQ_ERR_ARG; }
    init_chains_kernel<<<(h->n + 63) / 64, 64, 0, h->stream>>>(*h, s->dev());
    count_launch();
    MQ_CUDA(cudaGetLastError());
    h->models_set = true;
    return start_sampler_state(h, s);
}

// ---- desynchronised stepping -----------------------------------------------------------------------------------------
// Chains are independent, so nothing obliges them to advance in lock-step.  In a lock-step pass of a mixed proposal
// string only the chains that drew a velocity-model proposal (5 of 24 with the Example string) rebuild tables: the
// eikonal launch is a fifth full and the pass lasts as long as one warp-task.  Here a chain runs through its cheap
// proposals (hypocentre, station correction, noise) pass by pass until it draws one that needs tables, then parks;
// when most chains are parked one pass builds all their tables in a single full launch, decides them and sets them
// going again.  Every chain draws from its own counter-based stream, so its trajectory is the lock-step one, bit for
// bit (tests/test_sampler_gpu.py).  MCMCEQ_DESYNC=0 turns it off.
// true when every letter of the string is a proposal that rebuilds tables: nothing to run ahead with
static bool only_table_proposals(const char* str)
{
    if (!str || !*str) return false;
    for (const char* q = str; *q; q++)
        if (!strchr("PVMBD", *q)) return false;
    return true;
}

static bool desync_wanted(const Handle* h, int n_iters, const char* override_str)
{
    static int enabled = -1;
    if (enabled < 0) {
        const char* e = getenv("MCMCEQ_DESYNC");
        enabled = (e && e[0] == '0') ? 0 : 1;
    }
    if (override_str && *override_str) { if (only_table_proposals(override_str)) return false; }
    else if (only_table_proposals(h->cfg.dstring_start) && only_table_proposals(h->cfg.dstring_main)) return false;
    return enabled && n_iters >= 4 && h->cfg.eikonal == 1 && h->cfg.aflag != 1;
}

// The evaluate-and-decide part of every pass, behind the kernel that set up the proposal view `pv`: the table rebuilds
// that kernel queued (at most `items`; 0: it queued none), the misfit of every chain the view selects, the accept test and
// the records.
static int evaluate_and_decide(Handle* h, const EvalView& pv, const SamplerDev& d, int items)
{
    cudaStream_t st = h->stream;
    if (h->cfg.aflag != 1) {
        if (h->cfg.eikonal == 1 && items > 0) {
            MQ_CUDA(launch_rasterise(h, pv, items));
            MQ_CUDA(launch_tables(h, items));
        }
        MQ_CUDA(launch_misfit(h, pv));
        MQ_CUDA(launch_totals(h, pv));
    }
    accept_kernel<<<(h->n + 63) / 64, 64, 0, st>>>(*h, d, pv);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    snapshot_kernel<<<h->n, 128, 0, st>>>(*h, d);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    return MQ_OK;
}

static int step_desync(Handle* h, Sampler* s, int n_iters, int use_override)
{
    cudaStream_t st = h->stream;
    const int grid = (h->n + 63) / 64;
    const SamplerDev d = s->dev_desync();
    EvalView pv = h->prop_view;
    pv.hold = s->hold_buf;
    {
        std::vector<int32_t> todo((size_t)h->n, n_iters);
        MQ_CUDA(cudaMemcpyAsync(s->todo_buf, todo.data(), todo.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        MQ_CUDA(cudaMemsetAsync(s->hold_buf, 0, (size_t)h->n * sizeof(int32_t), st));
        MQ_CUDA(cudaStreamSynchronize(st));
    }
    int32_t stat[2] = {0, h->n};     // parked chains, chains that can still propose
    for (;;) {
        const int parked = stat[0], active = stat[1];
        if (parked == 0 && active == 0) break;
        // build tables when four fifths of the chains that are still at work wait for them, or nobody else can move
        const bool flush = parked > 0 && (active == 0 || 5L * parked >= 4L * (parked + active));
        MQ_CUDA(cudaMemsetAsync(s->stat_buf, 0, 2 * sizeof(int32_t), st));
        if (flush) {
            MQ_CUDA(cudaMemsetAsync(h->n_items, 0, sizeof(int32_t), st));
            flush_parked_kernel<<<grid, 64, 0, st>>>(*h, d, pv);
        } else {
            propose_kernel<<<grid, 64, 0, st>>>(*h, d, pv, use_override);   // parks the chains that need tables
        }
        count_launch();
        MQ_CUDA(cudaGetLastError());
        const int rc = evaluate_and_decide(h, pv, d, flush ? 2 * parked : 0);
        if (rc != MQ_OK) return rc;
        MQ_CUDA(cudaMemcpyAsync(stat, s->stat_buf, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        MQ_CUDA(cudaStreamSynchronize(st));
    }
    return check_device_errors(h);
}

extern "C" int mq_step(mq_handle* hh, int n_iters, const char* proposal_override)
{
    if (!hh || n_iters < 0) { set_error("mq_step: bad argument"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    if (!h->models_set) { set_error("mq_step: no models (mq_init_chains or mq_set_models first)"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    int rc = flags_poll(h, false);     // an error raised by the kernels of an earlier, asynchronous call
    if (rc != MQ_OK) return rc;
    Sampler* s;
    rc = started_sampler(h, &s);
    if (rc != MQ_OK) return rc;
    int use_override = 0;
    if (proposal_override && *proposal_override) {
        for (const char* q = proposal_override; *q; q++)
            if (!strchr("QRPVMBDN", *q)) { set_error("mq_step: unknown proposal letter '%c'", *q); return MQ_ERR_ARG; }
        if (s->over_host != proposal_override) {
            s->over_host = proposal_override;
            s->len_over = (int)s->over_host.size();
            MQ_CUDA(upload_string(&s->ps_over, s->over_host));
        }
        use_override = 1;
    }
    if (desync_wanted(h, n_iters, use_override ? proposal_override : nullptr)) return step_desync(h, s, n_iters, use_override);
    cudaStream_t st = h->stream;
    for (int it = 0; it < n_iters; it++) {
        MQ_CUDA(cudaMemsetAsync(h->n_items, 0, sizeof(int32_t), st));
        propose_kernel<<<(h->n + 63) / 64, 64, 0, st>>>(*h, s->dev(), h->prop_view, use_override);
        count_launch();
        MQ_CUDA(cudaGetLastError());
        rc = evaluate_and_decide(h, h->prop_view, s->dev(), 2 * h->n);
        if (rc != MQ_OK) return rc;
    }
    return n_iters > 0 ? flags_enqueue(h) : MQ_OK;   // stays asynchronous: reported by the next synchronising call
}

// Replay of a recorded proposal stream: see include/mcmceq_b200.h.
extern "C" int mq_replay_step(mq_handle* hh, const mq_replay* r)
{
    if (!hh || !r || !r->kind || !r->proposed || !r->u || !r->log_fac) { set_error("mq_replay_step: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    const mq_models* m = r->proposed;
    if (r->n_chains != h->n || m->n_chains != h->n || m->n_events != h->ne || m->n_stations != h->ns || m->max_dim < 1) {
        set_error("mq_replay_step: shape mismatch"); return MQ_ERR_ARG;
    }
    if (!h->models_set) { set_error("mq_replay_step: no models (mq_set_models or mq_init_chains first)"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    Sampler* s;
    int rc = started_sampler(h, &s);
    if (rc != MQ_OK) return rc;
    const size_t n = h->n, md = h->md, ne = h->ne, ns = h->ns;
    cudaStream_t st = h->stream;
    if (!h->prop_view.pres_over) { MQ_CUDA(dz(&h->prop_view.pres_over, n * ns)); MQ_CUDA(dz(&h->prop_view.sres_over, n * ns)); }
    // stage the injected proposal
    std::vector<int32_t> kind(n), dim(n), qidx(n, 0);
    std::vector<float> wz(n * md, 0.f), wvp(n * md, 1.f), wvs(n * md, 1.f), qxyz(3 * n, 0.f);
    for (size_t c = 0; c < n; c++) {
        kind[c] = (unsigned char)r->kind[c];
        if (kind[c] && !strchr("QRPVMBDN", kind[c])) { set_error("mq_replay_step: unknown proposal letter '%c'", kind[c]); return MQ_ERR_ARG; }
        dim[c] = m->dim[c];
        if (dim[c] < 1 || dim[c] > (int)md || dim[c] > m->max_dim) { set_error("mq_replay_step: chain %zu: %d nuclei", c, dim[c]); return MQ_ERR_ARG; }
        for (int i = 0; i < dim[c]; i++) {
            wz[c * md + i] = m->z[c * m->max_dim + i]; wvp[c * md + i] = m->vp[c * m->max_dim + i]; wvs[c * md + i] = m->vpvs[c * m->max_dim + i];
        }
        if (kind[c] == 'Q') {
            const int q = r->q_idx ? r->q_idx[c] : -1;
            if (q < 0 || q >= (int)ne) { set_error("mq_replay_step: chain %zu: event index %d", c, q); return MQ_ERR_ARG; }
            qidx[c] = q;
            for (int k = 0; k < 3; k++) qxyz[3 * c + k] = m->eq[(c * ne + q) * 3 + k];
        }
    }
    MQ_CUDA(cudaMemcpyAsync(s->kind, kind.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(s->r_qidx, qidx.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(s->r_dim, dim.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(s->wz, wz.data(), n * md * sizeof(float), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(s->wvp, wvp.data(), n * md * sizeof(float), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(s->wvs, wvs.data(), n * md * sizeof(float), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(h->prop_view.q_xyz, qxyz.data(), 3 * n * sizeof(float), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(h->prop_view.pres_over, m->pres, n * ns * sizeof(float), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(h->prop_view.sres_over, m->sres, n * ns * sizeof(float), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(s->noise_new, m->noise, n * 8 * sizeof(float), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(s->log_fac, r->log_fac, n * sizeof(double), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaMemcpyAsync(s->u_buf, r->u, n * sizeof(float), cudaMemcpyHostToDevice, st));
    MQ_CUDA(cudaStreamSynchronize(st));   // the staging vectors go out of scope below

    MQ_CUDA(cudaMemsetAsync(h->n_items, 0, sizeof(int32_t), st));
    const SamplerDev d = s->dev_replay();
    replay_setup_kernel<<<(h->n + 63) / 64, 64, 0, st>>>(*h, d, h->prop_view);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    rc = evaluate_and_decide(h, h->prop_view, d, 2 * h->n);
    if (rc != MQ_OK) return rc;
    if (r->accepted) MQ_CUDA(cudaMemcpyAsync(r->accepted, s->r_accept, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (r->alpha) MQ_CUDA(cudaMemcpyAsync(r->alpha, s->r_alpha, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (r->new_ll) MQ_CUDA(cudaMemcpyAsync(r->new_ll, s->r_newll, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (r->mf) MQ_CUDA(cudaMemcpyAsync(r->mf, h->mf_eval, n * 8 * sizeof(float), cudaMemcpyDeviceToHost, st));
    return check_device_errors(h);
}

extern "C" int mq_get_stats(mq_handle* hh, int64_t* counts, double* loglik, double* rms)
{
    if (!hh) { set_error("mq_get_stats: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    MQ_CUDA(cudaSetDevice(h->device));
    Sampler* s;
    int rc = sampler_get(h, &s);
    if (rc != MQ_OK) return rc;
    const size_t n = h->n;
    if (counts) MQ_CUDA(cudaMemcpyAsync(counts, s->counts, n * 20 * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    if (loglik) MQ_CUDA(cudaMemcpyAsync(loglik, h->ll, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (rms) MQ_CUDA(cudaMemcpyAsync(rms, h->rms, n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    MQ_CUDA(cudaStreamSynchronize(h->stream));
    return flags_poll(h, true);
}

// ---- records ---------------------------------------------------------------------------------
// Asynchronous path: mq_drain_begin enqueues, on the copy stream and behind everything the handle's stream holds so far,
// the pack kernel and the copy of its two counters; it returns at once, later steps run next to it.  mq_batch_wait (any
// host thread) waits for the counters, copies exactly the packed records into pinned memory and waits for them;
// mq_batch_deliver hands them to the callback.  Two batches exist per handle, so one can be written to disk while the
// next is being filled.
static void record_view(const float* rec, int md, int ne, int ns, mq_record* r)
{
    const int32_t* hi = (const int32_t*)rec;
    memset(r, 0, sizeof *r);
    r->chain = hi[0]; r->code = (char)hi[1]; r->dim = hi[2];
    memcpy(&r->number, rec + 4, sizeof(int64_t));
    memcpy(&r->rms, rec + 6, sizeof(double));
    const float* o = rec + kRecHead;
    r->noise = o; o += 8;
    r->z = o; r->vp = o + md; r->vpvs = o + 2 * md; o += 3 * (size_t)md;
    r->eq = o; o += 3 * (size_t)ne;
    r->origin = o; o += ne;
    r->pres = o; r->sres = o + ns;
    r->kind = MQ_REC_MODEL;
}

extern "C" int mq_set_ring(mq_handle* hh, int slots)
{
    if (!hh || slots < 1 || slots > 64) { set_error("mq_set_ring: 1 <= slots <= 64"); return MQ_ERR_ARG; }
    if (hh->h.sampler) { set_error("mq_set_ring: call before mq_init_chains / mq_step"); return MQ_ERR_STATE; }
    hh->h.ring_slots = slots;
    return MQ_OK;
}

extern "C" int mq_drain_begin(mq_handle* hh, mq_batch** out)
{
    if (!hh || !out) { set_error("mq_drain_begin: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    MQ_CUDA(cudaSetDevice(h->device));
    Sampler* s;
    int rc = sampler_get(h, &s);
    if (rc != MQ_OK) return rc;
    mq_batch* b = nullptr;
    for (int i = 0; i < 2 && !b; i++)
        if (s->batch[i].state == 0) b = &s->batch[i];
    if (!b) { set_error("mq_drain_begin: both batches are in flight (mq_batch_release one first)"); return MQ_ERR_BUSY; }
    if (!b->d_stage) {
        b->h = h;
        b->rec_floats = s->ring.rec_floats;
        b->cap_records = h->n * s->ring.slots;
        MQ_CUDA(cudaMalloc(&b->d_stage, (size_t)b->cap_records * b->rec_floats * sizeof(float)));
        MQ_CUDA(cudaMalloc(&b->d_count, 2 * sizeof(int32_t)));
        MQ_CUDA(cudaHostAlloc((void**)&b->h_count, 2 * sizeof(int32_t), cudaHostAllocDefault));
        MQ_CUDA(cudaEventCreateWithFlags(&b->ev_count, cudaEventDisableTiming));
        MQ_CUDA(cudaEventCreateWithFlags(&b->ev_data, cudaEventDisableTiming));
    }
    cudaStream_t cs = s->copy_stream;
    MQ_CUDA(cudaEventRecord(s->ev_main, h->stream));
    MQ_CUDA(cudaStreamWaitEvent(cs, s->ev_main, 0));
    MQ_CUDA(cudaMemsetAsync(b->d_count, 0, 2 * sizeof(int32_t), cs));
    pack_records_kernel<<<h->n, 128, 0, cs>>>(h->n, s->ring, b->d_stage, b->cap_records, b->d_count);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    MQ_CUDA(cudaMemcpyAsync(b->h_count, b->d_count, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, cs));
    MQ_CUDA(cudaEventRecord(b->ev_count, cs));
    b->state = 1; b->n_records = 0; b->n_lost = 0; b->delivered = 0;
    *out = b;
    return MQ_OK;
}

extern "C" int mq_batch_wait(mq_batch* b, int* n_records, int* n_lost)
{
    if (!b || b->state == 0) { set_error("mq_batch_wait: no drain begun on this batch"); return MQ_ERR_STATE; }
    if (b->state == 1) {
        Handle* h = b->h;
        Sampler* s = (Sampler*)h->sampler;
        MQ_CUDA(cudaSetDevice(h->device));
        MQ_CUDA(cudaEventSynchronize(b->ev_count));
        b->n_records = b->h_count[0]; b->n_lost = b->h_count[1];
        if (b->n_records > 0) {
            const size_t need = (size_t)b->n_records * b->rec_floats;
            if (need > b->h_cap_floats) {
                if (b->h_stage) cudaFreeHost(b->h_stage);
                b->h_stage = nullptr; b->h_cap_floats = 0;
                const size_t cap = std::max(need + need / 2, (size_t)1 << 18);
                MQ_CUDA(cudaHostAlloc((void**)&b->h_stage, cap * sizeof(float), cudaHostAllocDefault));
                b->h_cap_floats = cap;
            }
            MQ_CUDA(cudaMemcpyAsync(b->h_stage, b->d_stage, need * sizeof(float), cudaMemcpyDeviceToHost, s->copy_stream));
            MQ_CUDA(cudaEventRecord(b->ev_data, s->copy_stream));
            MQ_CUDA(cudaEventSynchronize(b->ev_data));
        }
        b->state = 2;
    }
    if (n_records) *n_records = b->n_records;
    if (n_lost) *n_lost = b->n_lost;
    return MQ_OK;
}

extern "C" int mq_batch_deliver(mq_batch* b, mq_record_fn fn, void* user)
{
    if (!b || !fn) { set_error("mq_batch_deliver: null"); return MQ_ERR_ARG; }
    if (b->state != 2) { const int rc = mq_batch_wait(b, nullptr, nullptr); if (rc != MQ_OK) return rc; }
    const Handle* h = b->h;
    // the pack kernel places the chains in the order its blocks arrive; deliver by chain number (a chain's records are
    // next to each other in the order they were produced, and the sort is stable)
    if (!b->order) b->order = new std::vector<int>();
    std::vector<int>& order = *b->order;
    if (b->delivered == 0) {
        order.resize((size_t)b->n_records);
        for (int i = 0; i < b->n_records; i++) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](int x, int y) {
            return ((const int32_t*)(b->h_stage + (size_t)x * b->rec_floats))[0] < ((const int32_t*)(b->h_stage + (size_t)y * b->rec_floats))[0];
        });
    }
    // a callback that returns non-zero stops the delivery; the records not yet delivered stay in the batch and a further
    // mq_batch_deliver call goes on with them (mq_batch_release discards them)
    while (b->delivered < b->n_records) {
        mq_record r;
        record_view(b->h_stage + (size_t)order[b->delivered] * b->rec_floats, h->md, h->ne, h->ns, &r);
        b->delivered++;
        if (fn(user, &r)) break;
    }
    return MQ_OK;
}

extern "C" int mq_batch_release(mq_batch* b)
{
    if (!b) return MQ_ERR_ARG;
    if (b->state == 1) { const int rc = mq_batch_wait(b, nullptr, nullptr); if (rc != MQ_OK) return rc; }
    b->state = 0;
    return MQ_OK;
}

extern "C" int mq_drain(mq_handle* hh, mq_record_fn fn, void* user, int* n_lost)
{
    if (!hh || !fn) { set_error("mq_drain: null"); return MQ_ERR_ARG; }
    mq_batch* b = nullptr;
    int rc = mq_drain_begin(hh, &b);
    if (rc != MQ_OK) return rc;
    int lost = 0;
    rc = mq_batch_wait(b, nullptr, &lost);
    if (rc == MQ_OK) rc = mq_batch_deliver(b, fn, user);
    mq_batch_release(b);
    if (n_lost) *n_lost = lost;
    if (rc != MQ_OK) return rc;
    return flags_poll(&hh->h, false);
}

// Copies of whole SoA arrays, then one callback per chain: 13 transfers whatever the number of chains.
static int deliver_soa(Handle* h, int first, int count, int kind, char code, const Snapshot& d, mq_record_fn fn, void* user)
{
    const size_t md = h->md, ne = h->ne, ns = h->ns, k = (size_t)count, c0 = (size_t)first;
    std::vector<int32_t> dim(k), cd(k);
    std::vector<int64_t> number(k);
    std::vector<double> rms(k);
    std::vector<float> z(k * md), vp(k * md), vpvs(k * md), eq(k * ne * 3), origin(k * ne), pres(k * ns), sres(k * ns), noise(k * 8);
    cudaStream_t st = h->stream;
#define D2H(dst, src, off, cnt) MQ_CUDA(cudaMemcpyAsync((dst).data(), (src) + (off), (cnt) * sizeof((dst)[0]), cudaMemcpyDeviceToHost, st))
    D2H(dim, d.dim, c0, k); D2H(cd, d.code, c0, k); D2H(number, d.number, c0, k); D2H(rms, d.rms, c0, k);
    D2H(z, d.z, c0 * md, k * md); D2H(vp, d.vp, c0 * md, k * md); D2H(vpvs, d.vpvs, c0 * md, k * md);
    D2H(eq, d.eq, c0 * ne * 3, k * ne * 3); D2H(origin, d.origin, c0 * ne, k * ne);
    D2H(pres, d.pres, c0 * ns, k * ns); D2H(sres, d.sres, c0 * ns, k * ns); D2H(noise, d.noise, c0 * 8, k * 8);
#undef D2H
    MQ_CUDA(cudaStreamSynchronize(st));
    for (size_t i = 0; i < k; i++) {
        mq_record r;
        memset(&r, 0, sizeof r);
        r.chain = (int)(c0 + i); r.kind = kind; r.code = code ? code : (char)cd[i]; r.number = number[i]; r.dim = dim[i]; r.rms = rms[i];
        r.z = &z[i * md]; r.vp = &vp[i * md]; r.vpvs = &vpvs[i * md]; r.eq = &eq[i * ne * 3]; r.origin = &origin[i * ne];
        r.pres = &pres[i * ns]; r.sres = &sres[i * ns]; r.noise = &noise[i * 8];
        if (fn(user, &r)) break;
    }
    return MQ_OK;
}

// gathers the current state of every chain (current model / origin buffers) into the layout of a Snapshot
__global__ void gather_current_kernel(Handle hd, SamplerDev s, Snapshot d)
{
    const int c = blockIdx.x;
    snapshot_copy(hd, d, c);
    if (threadIdx.x == 0) {
        const int64_t acce = s.acce[c];
        d.number[c] = acce > 0 ? acce - 1 : 0;
        d.rms[c] = hd.rms[c];
        d.code[c] = 'S';
    }
}

static int snapshot_range(mq_handle* hh, int first, int count, int which, mq_record_fn fn, void* user)
{
    Handle* h = &hh->h;
    MQ_CUDA(cudaSetDevice(h->device));
    Sampler* s;
    int rc = sampler_get(h, &s);
    if (rc != MQ_OK) return rc;
    if (which == 1) return deliver_soa(h, first, count, MQ_REC_BEST, 'F', s->best, fn, user);
    // current state: gathered on the device into a scratch snapshot, then the same bulk copies
    if (!s->cur.dim) MQ_CUDA(alloc_snapshot(&s->cur, h));
    gather_current_kernel<<<h->n, 128, 0, h->stream>>>(*h, s->dev(), s->cur);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    return deliver_soa(h, first, count, MQ_REC_CURRENT, 'S', s->cur, fn, user);
}

extern "C" int mq_snapshot(mq_handle* hh, int chain, int which, mq_record_fn fn, void* user)
{
    if (!hh || !fn || chain < 0 || chain >= hh->h.n || which < 0 || which > 1) { set_error("mq_snapshot: bad argument"); return MQ_ERR_ARG; }
    return snapshot_range(hh, chain, 1, which, fn, user);
}

extern "C" int mq_snapshot_all(mq_handle* hh, int which, mq_record_fn fn, void* user)
{
    if (!hh || !fn || which < 0 || which > 1) { set_error("mq_snapshot_all: bad argument"); return MQ_ERR_ARG; }
    return snapshot_range(hh, 0, hh->h.n, which, fn, user);
}
