// hypo.cu -- hypocentre uncertainty on the device: per event the mean and 4 x 4 covariance of (x, y, z, t), quantiles and
// mode of x, y and z, and the error ellipsoid (mq_hypo_begin, mq_hypo_chains, mq_hypo_summary; DESIGN.md section 4e).
//
// snapshot_kernel (chain.cu, hypo_accumulate) adds every used decimated model to per-(chain, event) sums of d = v - ref
// and of the products d_i d_j, and to per-event histograms of x, y and z.  The summary reduces the sums over chains in a
// fixed order -- events across threads, chains split into a fixed number of groups that depends on the chain and event
// counts only, groups combined in order -- with no floating-point atomics: the same accumulators always give the same
// bits.  Round 1 gives N, the mean and the pooled within-chain scatter, round 2 the between-chain scatter about that mean;
// across ranks each round's sums are all-reduced, and the histograms as int32.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../include/mcmceq_b200.h"
#include "chain.cuh"
#include "errors.h"
#include "launch_count.h"
#include "state.h"

namespace mq {

// diag.cu: tot[j][q] = sum over g, group 0 first, of part[g][j][q]
__global__ void diag_combine_kernel(const double* part, int groups, int rows, int Q, double* tot);

constexpr int kHypoThreads = 128;
constexpr int kHypoBlocks = 1184;   // 8 blocks per SM of a B200; only the group count follows from it, not the device
constexpr int kRound1 = 15;         // partial sums per event: N, sum of n_c ref_c + S_c [4], sum of W_c [10]
constexpr int kRound2 = 10;         // sum of n_c (m_c - mean)_i (m_c - mean)_j [10]
constexpr int kOut = 50;            // doubles out per event: mean 4 | cov 16 | quant 15 | mode 3 | axes 3 | axis_dir 9
constexpr int kMaxBins = 1 << 20;
constexpr int kJacobiSweeps = 32;
__constant__ double kProb[5] = {0.025, 0.16, 0.5, 0.84, 0.975};

struct HypoPlan {
    int xb, groups, per_group;
    size_t part1, tot1, part2, tot2, out, doubles;   // offsets in the scratch (doubles)
    size_t hist_bytes, bytes;                        // a copy of the histograms after the doubles (collective only)
};

static HypoPlan hypo_plan(int n, int ne, int nbt)
{
    HypoPlan P;
    P.xb = (ne + kHypoThreads - 1) / kHypoThreads;
    int g = (kHypoBlocks + P.xb - 1) / P.xb;
    if (g > n) g = n;
    if (g < 1) g = 1;
    P.per_group = (n + g - 1) / g;
    P.groups = (n + P.per_group - 1) / P.per_group;
    const size_t e = (size_t)ne;
    P.part1 = 0;
    P.tot1 = P.part1 + (size_t)P.groups * kRound1 * e;
    P.part2 = P.tot1 + kRound1 * e;
    P.tot2 = P.part2 + (size_t)P.groups * kRound2 * e;
    P.out = P.tot2 + kRound2 * e;
    P.doubles = P.out + kOut * e;
    P.hist_bytes = e * nbt * sizeof(int32_t);
    P.bytes = P.doubles * sizeof(double) + P.hist_bytes;
    return P;
}

// Round 1, one thread per (event, chain group): over the group's chains in order, N, sum (n_c ref_c + S_c) and the
// within-chain scatter W_c = C_c - S_c[i] S_c[j] / n_c.
__global__ void __launch_bounds__(kHypoThreads) hypo_chains_kernel(Hypo H, int n, int ne, int per_group, double* part)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= ne) return;
    const int c0 = blockIdx.y * per_group, c1 = min(n, c0 + per_group);
    double a[kRound1];
    for (int j = 0; j < kRound1; j++) a[j] = 0.0;
    for (int c = c0; c < c1; c++) {
        const double nc = (double)H.n_models[c];
        if (nc == 0.0) continue;
        double S[4];
        for (int k = 0; k < 4; k++) {
            S[k] = H.sum[((size_t)c * 4 + k) * ne + e];
            const double ref = H.ref[((size_t)c * 4 + k) * ne + e];
            a[1 + k] = __dadd_rn(a[1 + k], __dadd_rn(__dmul_rn(nc, ref), S[k]));
        }
        a[0] = __dadd_rn(a[0], nc);
        int p = 0;
        for (int i = 0; i < 4; i++)
            for (int j = i; j < 4; j++, p++) {
                const double w = __dsub_rn(H.cross[((size_t)c * 10 + p) * ne + e], __ddiv_rn(__dmul_rn(S[i], S[j]), nc));
                a[5 + p] = __dadd_rn(a[5 + p], w);
            }
    }
    for (int j = 0; j < kRound1; j++) part[((size_t)blockIdx.y * kRound1 + j) * ne + e] = a[j];
}

// Round 2, per (event, chain group): the between-chain scatter n_c (m_c - mean)(m_c - mean)^T, m_c = ref_c + S_c / n_c.
__global__ void __launch_bounds__(kHypoThreads) hypo_spread_kernel(Hypo H, int n, int ne, int per_group, const double* tot1,
                                                                  double* part2)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= ne) return;
    const int c0 = blockIdx.y * per_group, c1 = min(n, c0 + per_group);
    const double N = tot1[e];
    double mu[4], b[kRound2];
    for (int k = 0; k < 4; k++) mu[k] = __ddiv_rn(tot1[(size_t)(1 + k) * ne + e], N);
    for (int j = 0; j < kRound2; j++) b[j] = 0.0;
    for (int c = c0; c < c1; c++) {
        const double nc = (double)H.n_models[c];
        if (nc == 0.0) continue;
        double d[4];
        for (int k = 0; k < 4; k++) {
            const double m = __dadd_rn(H.ref[((size_t)c * 4 + k) * ne + e], __ddiv_rn(H.sum[((size_t)c * 4 + k) * ne + e], nc));
            d[k] = __dsub_rn(m, mu[k]);
        }
        int p = 0;
        for (int i = 0; i < 4; i++)
            for (int j = i; j < 4; j++, p++) b[p] = __dadd_rn(b[p], __dmul_rn(nc, __dmul_rn(d[i], d[j])));
    }
    for (int j = 0; j < kRound2; j++) part2[((size_t)blockIdx.y * kRound2 + j) * ne + e] = b[j];
}

// Eigen-decomposition of a symmetric 3 x 3 matrix by cyclic Jacobi rotations: a ends diagonal (the eigenvalues), the
// columns of v are the eigenvectors.  hypo.py restates it operation for operation.
__device__ void jacobi3(double a[3][3], double v[3][3])
{
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) v[i][j] = i == j ? 1.0 : 0.0;
    const int P[3] = {0, 0, 1}, Qi[3] = {1, 2, 2};
    for (int sweep = 0; sweep < kJacobiSweeps; sweep++) {
        if (a[0][1] == 0.0 && a[0][2] == 0.0 && a[1][2] == 0.0) break;
#pragma unroll
        for (int r = 0; r < 3; r++) {
            const int p = P[r], q = Qi[r], o = 3 - p - q;
            const double apq = a[p][q];
            if (apq == 0.0) continue;
            const double g = 100.0 * fabs(apq);
            if (sweep > 3 && fabs(a[p][p]) + g == fabs(a[p][p]) && fabs(a[q][q]) + g == fabs(a[q][q])) {
                a[p][q] = a[q][p] = 0.0;   // negligible against both diagonal entries
                continue;
            }
            const double hd = a[q][q] - a[p][p];
            double t;
            if (fabs(hd) + g == fabs(hd)) {
                t = apq / hd;
            } else {
                const double theta = 0.5 * hd / apq;
                t = 1.0 / (fabs(theta) + sqrt(1.0 + theta * theta));
                if (theta < 0.0) t = -t;
            }
            const double c = 1.0 / sqrt(1.0 + t * t), s = t * c, tau = s / (1.0 + c), h = t * apq;
            a[p][p] -= h;
            a[q][q] += h;
            a[p][q] = a[q][p] = 0.0;
            const double gp = a[o][p], gq = a[o][q];
            a[o][p] = a[p][o] = gp - s * (gq + gp * tau);
            a[o][q] = a[q][o] = gq + s * (gp - gq * tau);
            for (int k = 0; k < 3; k++) {
                const double vp = v[k][p], vq = v[k][q];
                v[k][p] = vp - s * (vq + vp * tau);
                v[k][q] = vq + s * (vp - vq * tau);
            }
        }
    }
}

// Per event from the job-wide sums: mean, covariance and the error ellipsoid of the spatial block.
__global__ void __launch_bounds__(kHypoThreads) hypo_final_kernel(int ne, const double* tot1, const double* tot2, double* out)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= ne) return;
    double* o = out + (size_t)e * kOut;
    const double N = tot1[e];
    double cov[4][4];
    int p = 0;
    for (int i = 0; i < 4; i++) {
        o[i] = N > 0.0 ? __ddiv_rn(tot1[(size_t)(1 + i) * ne + e], N) : NAN;
        for (int j = i; j < 4; j++, p++) {
            const double s = __dadd_rn(tot1[(size_t)(5 + p) * ne + e], tot2[(size_t)p * ne + e]);
            cov[i][j] = cov[j][i] = N > 1.0 ? __ddiv_rn(s, N - 1.0) : NAN;
        }
    }
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) o[4 + 4 * i + j] = cov[i][j];
    double* axes = o + 38;
    double* dir = o + 41;
    if (!(N > 1.0)) {
        for (int k = 0; k < 12; k++) axes[k] = NAN;   // axes and axis_dir
        return;
    }
    double a[3][3], v[3][3];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) a[i][j] = cov[i][j];
    jacobi3(a, v);
    int ord[3] = {0, 1, 2};   // descending eigenvalue, the lower index first on a tie
    for (int i = 0; i < 2; i++)
        for (int j = 0; j < 2 - i; j++)
            if (a[ord[j + 1]][ord[j + 1]] > a[ord[j]][ord[j]]) { const int t = ord[j]; ord[j] = ord[j + 1]; ord[j + 1] = t; }
    for (int k = 0; k < 3; k++) {
        const int c = ord[k];
        const double lam = a[c][c];
        axes[k] = lam > 0.0 ? sqrt(lam) : 0.0;
        double x = v[0][c], y = v[1][c], z = v[2][c];
        if (z < 0.0 || (z == 0.0 && (y < 0.0 || (y == 0.0 && x < 0.0)))) { x = -x; y = -y; z = -z; }
        dir[3 * k] = x; dir[3 * k + 1] = y; dir[3 * k + 2] = z;
    }
}

// Quantiles and mode of one (event, axis) histogram per warp: a running integer prefix scan over the bins, 32 at a time.
__global__ void __launch_bounds__(kHypoThreads) hypo_quant_kernel(const int32_t* hist, int ne, int nb0, int nb1, int nb2, float lo0,
                                                                 float lo1, float lo2, float w, double* out)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int wi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (wi >= 3 * ne) return;   // the whole warp
    const int e = wi / 3, ax = wi % 3;
    const int B = ax == 0 ? nb0 : ax == 1 ? nb1 : nb2;
    const int32_t* h = hist + (size_t)e * (nb0 + nb1 + nb2) + (ax == 0 ? 0 : ax == 1 ? nb0 : nb0 + nb1);
    const double lo = ax == 0 ? lo0 : ax == 1 ? lo1 : lo2, wd = w;
    double* quant = out + (size_t)e * kOut + 20 + 5 * ax;
    double* mode = out + (size_t)e * kOut + 35 + ax;
    long long tot = 0;
    for (int j = lane; j < B; j += 32) tot += h[j];
    for (int s = 16; s > 0; s >>= 1) tot += __shfl_xor_sync(full, tot, s);
    if (tot == 0) {
        if (lane < 5) quant[lane] = NAN;
        if (lane == 0) *mode = NAN;
        return;
    }
    double target[5], res[5];
    for (int k = 0; k < 5; k++) { target[k] = __dmul_rn(kProb[k], (double)tot); res[k] = NAN; }
    int found = 0, best = -1, best_j = 0;
    long long base = 0;
    for (int j0 = 0; j0 < B; j0 += 32) {
        const int j = j0 + lane;
        const int cnt = j < B ? h[j] : 0;
        long long cum = cnt;
        for (int s = 1; s < 32; s <<= 1) {
            const long long t = __shfl_up_sync(full, cum, s);
            if (lane >= s) cum += t;
        }
        cum += base;
        if (j < B && cnt > best) { best = cnt; best_j = j; }   // bins ascending per lane: the first of equal counts stays
        for (int k = 0; k < 5; k++) {
            if (found & (1 << k)) continue;
            const unsigned b = __ballot_sync(full, j < B && (double)cum >= target[k]);
            if (b) {
                const int l = __ffs(b) - 1;
                const long long cl = __shfl_sync(full, cum, l);
                const int cn = __shfl_sync(full, cnt, l);
                const double frac = __ddiv_rn(__dsub_rn(target[k], (double)(cl - cn)), (double)cn);
                res[k] = __dadd_rn(lo, __dmul_rn(wd, __dadd_rn((double)(j0 + l), frac)));
                found |= 1 << k;
            }
        }
        base = __shfl_sync(full, cum, 31);
    }
    for (int s = 16; s > 0; s >>= 1) {
        const int ob = __shfl_xor_sync(full, best, s), oj = __shfl_xor_sync(full, best_j, s);
        if (ob > best || (ob == best && oj < best_j)) { best = ob; best_j = oj; }
    }
    for (int k = 0; k < 5; k++)
        if (lane == k) quant[k] = res[k];
    if (lane == 0) *mode = __dadd_rn(lo, __dmul_rn(wd, (double)best_j + 0.5));
}

int hypo_bins(const Handle* h, float bin_km, int nb[3])
{
    const float lo[3] = {h->xmin, h->ymin, h->zmin}, hi[3] = {h->xmax, h->ymax, h->zmax};
    for (int a = 0; a < 3; a++) {
        const float span = hi[a] - lo[a];
        const float q = span / bin_km;
        if (!(q < (float)kMaxBins)) return -1;   // also NaN
        nb[a] = (int)q + 1;
    }
    return 0;
}

int hypo_alloc(Handle* h, float bin_km, long long burn_in)
{
    hypo_destroy(h);
    Hypo& H = h->hypo;
    if (hypo_bins(h, bin_km, H.nb) != 0) return MQ_ERR_ARG;
    H.bin = bin_km;
    H.burn_in = burn_in;
    const size_t n = h->n, ne = h->ne, nbt = (size_t)H.nb[0] + H.nb[1] + H.nb[2];
    MQ_CUDA(cudaMalloc((void**)&H.hist, ne * nbt * sizeof(int32_t)));
    MQ_CUDA(cudaMalloc((void**)&H.outside, ne * 3 * sizeof(int32_t)));
    MQ_CUDA(cudaMalloc((void**)&H.ref, n * 4 * ne * sizeof(double)));
    MQ_CUDA(cudaMalloc((void**)&H.sum, n * 4 * ne * sizeof(double)));
    MQ_CUDA(cudaMalloc((void**)&H.cross, n * 10 * ne * sizeof(double)));
    MQ_CUDA(cudaMalloc((void**)&H.n_models, n * sizeof(int64_t)));
    cudaStream_t st = h->stream;
    MQ_CUDA(cudaMemsetAsync(H.hist, 0, ne * nbt * sizeof(int32_t), st));
    MQ_CUDA(cudaMemsetAsync(H.outside, 0, ne * 3 * sizeof(int32_t), st));
    MQ_CUDA(cudaMemsetAsync(H.ref, 0, n * 4 * ne * sizeof(double), st));
    MQ_CUDA(cudaMemsetAsync(H.sum, 0, n * 4 * ne * sizeof(double), st));
    MQ_CUDA(cudaMemsetAsync(H.cross, 0, n * 10 * ne * sizeof(double), st));
    MQ_CUDA(cudaMemsetAsync(H.n_models, 0, n * sizeof(int64_t), st));
    H.on = 1;
    return MQ_OK;
}

void hypo_destroy(Handle* h)
{
    Hypo& H = h->hypo;
    if (H.hist || H.scratch) {
        cudaSetDevice(h->device);
        if (h->stream) cudaStreamSynchronize(h->stream);
    }
    cudaFree(H.hist); cudaFree(H.outside); cudaFree(H.ref); cudaFree(H.sum); cudaFree(H.cross); cudaFree(H.n_models);
    cudaFree(H.scratch);
    memset(&H, 0, sizeof H);
}

}  // namespace mq

using namespace mq;

extern "C" int mq_hypo_begin(mq_handle* hh, float bin_km, int64_t burn_in, mq_hypo_dims* dims)
{
    if (!hh) { set_error("mq_hypo_begin: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    int nb[3];
    if (!(bin_km > 0.f) || burn_in < 0 || hypo_bins(h, bin_km, nb) != 0) {
        set_error("mq_hypo_begin: bin width %g km, burn_in %lld (bin width > 0 and at most 2^20 bins per axis; burn_in >= 0)",
                  (double)bin_km, (long long)burn_in);
        return MQ_ERR_ARG;
    }
    MQ_CUDA(cudaSetDevice(h->device));
    const int rc = hypo_alloc(h, bin_km, (long long)burn_in);
    if (rc != MQ_OK) { hypo_destroy(h); return rc; }
    if (dims) {
        dims->n_events = h->ne;
        dims->bin_km = bin_km;
        for (int a = 0; a < 3; a++) dims->n_bins[a] = h->hypo.nb[a];
        dims->lo[0] = h->xmin; dims->lo[1] = h->ymin; dims->lo[2] = h->zmin;
    }
    return MQ_OK;
}

extern "C" int mq_hypo_chains(mq_handle* hh, int32_t* hist, int32_t* outside, double* ref, double* sum, double* cross, int64_t* n_models)
{
    if (!hh) { set_error("mq_hypo_chains: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    const Hypo& H = h->hypo;
    if (!H.on) { set_error("mq_hypo_chains: mq_hypo_begin was not called"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    int rc = flags_poll(h, true);
    if (rc != MQ_OK) return rc;
    cudaStream_t s = h->stream;
    const size_t n = h->n, ne = h->ne, nbt = (size_t)H.nb[0] + H.nb[1] + H.nb[2];
#define GET(dst, src, cnt) if (dst) MQ_CUDA(cudaMemcpyAsync(dst, src, (cnt) * sizeof(*(dst)), cudaMemcpyDeviceToHost, s))
    GET(hist, H.hist, ne * nbt); GET(outside, H.outside, ne * 3);
    GET(ref, H.ref, n * 4 * ne); GET(sum, H.sum, n * 4 * ne); GET(cross, H.cross, n * 10 * ne); GET(n_models, H.n_models, n);
#undef GET
    MQ_CUDA(cudaStreamSynchronize(s));
    return check_device_errors(h);
}

extern "C" int mq_hypo_summary(mq_handle* hh, int collective, double* mean, double* cov, double* quant, double* mode, double* axes,
                               double* axis_dir, int64_t* n_models)
{
    if (!hh) { set_error("mq_hypo_summary: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    Hypo& H = h->hypo;
    MQ_CUDA(cudaSetDevice(h->device));
    int rc = flags_poll(h, true);     // an error of an earlier asynchronous call comes first
    if (rc != MQ_OK) return rc;
    if (!H.on) { set_error("mq_hypo_summary: mq_hypo_begin was not called"); return MQ_ERR_STATE; }
    const int ne = h->ne, n = h->n, nbt = H.nb[0] + H.nb[1] + H.nb[2];
    const HypoPlan P = hypo_plan(n, ne, nbt);
    if (H.scratch_bytes < P.bytes) {
        cudaFree(H.scratch);
        H.scratch = nullptr; H.scratch_bytes = 0;
        MQ_CUDA(cudaMalloc(&H.scratch, P.bytes));
        H.scratch_bytes = P.bytes;
    }
    double* w = (double*)H.scratch;
    cudaStream_t st = h->stream;
    const dim3 grid_g(P.xb, P.groups), grid_e(P.xb);
    hypo_chains_kernel<<<grid_g, kHypoThreads, 0, st>>>(H, n, ne, P.per_group, w + P.part1);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    diag_combine_kernel<<<grid_e, kHypoThreads, 0, st>>>(w + P.part1, P.groups, kRound1, ne, w + P.tot1);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    if (collective) { rc = comm_allreduce_sum(h, w + P.tot1, kRound1 * (size_t)ne); if (rc != MQ_OK) return rc; }
    hypo_spread_kernel<<<grid_g, kHypoThreads, 0, st>>>(H, n, ne, P.per_group, w + P.tot1, w + P.part2);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    diag_combine_kernel<<<grid_e, kHypoThreads, 0, st>>>(w + P.part2, P.groups, kRound2, ne, w + P.tot2);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    if (collective) { rc = comm_allreduce_sum(h, w + P.tot2, kRound2 * (size_t)ne); if (rc != MQ_OK) return rc; }
    hypo_final_kernel<<<grid_e, kHypoThreads, 0, st>>>(ne, w + P.tot1, w + P.tot2, w + P.out);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    const int32_t* hist = H.hist;
    if (collective) {   // the job-wide histograms in the work space; the handle's own stay as they are
        int32_t* all = (int32_t*)(w + P.doubles);
        MQ_CUDA(cudaMemcpyAsync(all, H.hist, P.hist_bytes, cudaMemcpyDeviceToDevice, st));
        rc = comm_allreduce_sum(h, all, P.hist_bytes / sizeof(int32_t));
        if (rc != MQ_OK) return rc;
        hist = all;
    }
    const int warps_per_block = kHypoThreads / 32;
    hypo_quant_kernel<<<(3 * ne + warps_per_block - 1) / warps_per_block, kHypoThreads, 0, st>>>(
        hist, ne, H.nb[0], H.nb[1], H.nb[2], h->xmin, h->ymin, h->zmin, H.bin, w + P.out);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    std::vector<double> out((size_t)kOut * ne);
    double total = 0.0;
    MQ_CUDA(cudaMemcpyAsync(out.data(), w + P.out, out.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    MQ_CUDA(cudaMemcpyAsync(&total, w + P.tot1, sizeof(double), cudaMemcpyDeviceToHost, st));   // N of event 0 = N of all
    MQ_CUDA(cudaStreamSynchronize(st));
    for (int e = 0; e < ne; e++) {
        const double* o = out.data() + (size_t)e * kOut;
        if (mean) memcpy(mean + 4 * (size_t)e, o, 4 * sizeof(double));
        if (cov) memcpy(cov + 16 * (size_t)e, o + 4, 16 * sizeof(double));
        if (quant) memcpy(quant + 15 * (size_t)e, o + 20, 15 * sizeof(double));
        if (mode) memcpy(mode + 3 * (size_t)e, o + 35, 3 * sizeof(double));
        if (axes) memcpy(axes + 3 * (size_t)e, o + 38, 3 * sizeof(double));
        if (axis_dir) memcpy(axis_dir + 9 * (size_t)e, o + 41, 9 * sizeof(double));
    }
    if (n_models) *n_models = (int64_t)(total + 0.5);
    return check_device_errors(h);
}
