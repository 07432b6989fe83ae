// diag.cu -- convergence diagnostics on the device: split R-hat and batch-means effective sample size of every quantity
// the posterior summarises (mq_diag_begin, mq_diag_chains, mq_diag_summary; DESIGN.md section 4d).
//
// snapshot_kernel (chain.cu, diag_accumulate) adds every used decimated model of a chain to K batch slots of sums of
// d = x - ref and of d*d, per quantity; when all K slots are full, pairs merge and the batch length doubles.  The summary
// reduces those accumulators over chains in a fixed order -- quantities across threads, chains split into a fixed number
// of groups that depends on the chain and quantity counts only, groups combined in order -- with no floating-point
// atomics: the same accumulators always give the same bits.  Across ranks the partial sums are all-reduced in two rounds
// (the sums that give the mean of the sequence means, then the squared deviations from it).
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

constexpr int kDiagThreads = 128;
constexpr int kDiagBlocks = 1184;   // 8 blocks per SM of a B200; only the group count follows from it, not the device
constexpr int kParts = 8;           // partial sums per quantity, in this order:
// chains used, sum of s_j^2, sum of mu_j, sum of n_j, sum of L_c sum_b (y_cb - ybar_c)^2, sum of (k_c - 1), N = sum k_c L_c,
// sum of k_c L_c ref_c + sum_b S_cb

struct DiagPlan {
    int xb, groups, per_group;
    size_t part, tot1, part2, tot2, out, mu, doubles;   // offsets in the scratch (doubles)
};

static DiagPlan diag_plan(int n, int Q)
{
    DiagPlan P;
    P.xb = (Q + kDiagThreads - 1) / kDiagThreads;
    int g = (kDiagBlocks + P.xb - 1) / P.xb;
    if (g > n) g = n;
    if (g < 1) g = 1;
    P.per_group = (n + g - 1) / g;
    P.groups = (n + P.per_group - 1) / P.per_group;
    const size_t q = (size_t)Q;
    P.part = 0;
    P.tot1 = P.part + (size_t)P.groups * kParts * q;
    P.part2 = P.tot1 + kParts * q;
    P.tot2 = P.part2 + (size_t)P.groups * q;
    P.out = P.tot2 + q;
    P.mu = P.out + 4 * q;
    P.doubles = P.mu + 2 * (size_t)n * q;
    return P;
}

// Pass 1, one thread per (quantity, chain group): the per-chain statistics of every chain of the group with k_c >= 4, in
// chain order, and the two sequence means mu_j of each chain (kept for pass 3).
__global__ void __launch_bounds__(kDiagThreads) diag_chains_kernel(Diag D, int n, int per_group, double* part, double* mu)
{
    const int Q = D.Q, K = D.K;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    const int c0 = blockIdx.y * per_group, c1 = min(n, c0 + per_group);
    double a[kParts];
    for (int j = 0; j < kParts; j++) a[j] = 0.0;
    for (int c = c0; c < c1; c++) {
        const int k = D.full_batches[c];
        if (k < 4) continue;
        const int L = D.batch_len[c], h = k / 2;
        const double* S = D.sum + (size_t)c * K * Q + q;
        const double* T = D.sumsq + (size_t)c * K * Q + q;
        const double ref = D.ref[(size_t)c * Q + q];
        double sa = 0.0, ta = 0.0, sb = 0.0, tb = 0.0, sall = 0.0, ysum = 0.0;
        for (int b = 0; b < k; b++) {
            const double s = S[(size_t)b * Q];
            if (b < h) { sa = __dadd_rn(sa, s); ta = __dadd_rn(ta, T[(size_t)b * Q]); }
            else if (b < 2 * h) { sb = __dadd_rn(sb, s); tb = __dadd_rn(tb, T[(size_t)b * Q]); }
            sall = __dadd_rn(sall, s);
            ysum = __dadd_rn(ysum, __ddiv_rn(s, (double)L));
        }
        const double ybar = __ddiv_rn(ysum, (double)k);
        double dev = 0.0;
        for (int b = 0; b < k; b++) {
            const double e = __dsub_rn(__ddiv_rn(S[(size_t)b * Q], (double)L), ybar);
            dev = __dadd_rn(dev, __dmul_rn(e, e));
        }
        const double nj = (double)h * (double)L;
        const double ma = __ddiv_rn(sa, nj), mb = __ddiv_rn(sb, nj);
        const double s2a = __ddiv_rn(__dsub_rn(ta, __dmul_rn(sa, ma)), nj - 1.0);
        const double s2b = __ddiv_rn(__dsub_rn(tb, __dmul_rn(sb, mb)), nj - 1.0);
        const double mua = __dadd_rn(ref, ma), mub = __dadd_rn(ref, mb);
        mu[((size_t)c * 2) * Q + q] = mua;
        mu[((size_t)c * 2 + 1) * Q + q] = mub;
        const double kl = (double)k * (double)L;
        a[0] = __dadd_rn(a[0], 1.0);
        a[1] = __dadd_rn(__dadd_rn(a[1], s2a), s2b);
        a[2] = __dadd_rn(__dadd_rn(a[2], mua), mub);
        a[3] = __dadd_rn(a[3], 2.0 * nj);
        a[4] = __dadd_rn(a[4], __dmul_rn((double)L, dev));
        a[5] = __dadd_rn(a[5], (double)(k - 1));
        a[6] = __dadd_rn(a[6], kl);
        a[7] = __dadd_rn(a[7], __dadd_rn(__dmul_rn(kl, ref), sall));
    }
    for (int j = 0; j < kParts; j++) part[((size_t)blockIdx.y * kParts + j) * Q + q] = a[j];
}

// sum over groups, group 0 first: tot[j][q] = sum_g part[g][j][q]
__global__ void __launch_bounds__(kDiagThreads) diag_combine_kernel(const double* part, int groups, int rows, int Q, double* tot)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    for (int j = 0; j < rows; j++) {
        double s = 0.0;
        for (int g = 0; g < groups; g++) s = __dadd_rn(s, part[((size_t)g * rows + j) * Q + q]);
        tot[(size_t)j * Q + q] = s;
    }
}

// Pass 3, per (quantity, chain group): sum of (mu_j - mubar)^2 over the sequences of the group's used chains.
__global__ void __launch_bounds__(kDiagThreads) diag_spread_kernel(Diag D, int n, int per_group, const double* tot1, const double* mu,
                                                                  double* part2)
{
    const int Q = D.Q;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    const int c0 = blockIdx.y * per_group, c1 = min(n, c0 + per_group);
    const double mubar = __ddiv_rn(tot1[2 * (size_t)Q + q], 2.0 * tot1[q]);
    double b = 0.0;
    for (int c = c0; c < c1; c++) {
        if (D.full_batches[c] < 4) continue;
        const double ea = __dsub_rn(mu[((size_t)c * 2) * Q + q], mubar), eb = __dsub_rn(mu[((size_t)c * 2 + 1) * Q + q], mubar);
        b = __dadd_rn(__dadd_rn(b, __dmul_rn(ea, ea)), __dmul_rn(eb, eb));
    }
    part2[(size_t)blockIdx.y * Q + q] = b;
}

// The summary of every quantity from the job-wide sums: out = mean [Q] | sd [Q] | rhat [Q] | ess [Q].
__global__ void __launch_bounds__(kDiagThreads) diag_final_kernel(int Q, const double* tot1, const double* tot2, double* out)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    const double used = tot1[q];
    double mean = NAN, sd = NAN, rhat = NAN, ess = NAN;
    if (used > 0.0) {
        const double M = 2.0 * used, N = tot1[6 * (size_t)Q + q];
        const double W = __ddiv_rn(tot1[(size_t)Q + q], M);
        const double Bv = __ddiv_rn(tot2[q], M - 1.0);
        const double nbar = __ddiv_rn(tot1[3 * (size_t)Q + q], M);
        const double varp = __dadd_rn(__dmul_rn(__ddiv_rn(nbar - 1.0, nbar), W), Bv);
        const double sig = __ddiv_rn(tot1[4 * (size_t)Q + q], tot1[5 * (size_t)Q + q]);
        mean = __ddiv_rn(tot1[7 * (size_t)Q + q], N);
        sd = __dsqrt_rn(varp);
        if (varp > 0.0) {
            rhat = W > 0.0 ? __dsqrt_rn(__ddiv_rn(varp, W)) : INFINITY;
            ess = sig > 0.0 ? __ddiv_rn(__dmul_rn(N, varp), sig) : INFINITY;
        }
    }
    out[q] = mean;
    out[(size_t)Q + q] = sd;
    out[2 * (size_t)Q + q] = rhat;
    out[3 * (size_t)Q + q] = ess;
}

int diag_alloc(Handle* h, int K, long long burn_in)
{
    diag_destroy(h);
    Diag& D = h->diag;
    const size_t n = h->n;
    D.K = K;
    D.Q = diag_quantities(h->nz, h->ne, h->ns);
    D.burn_in = burn_in;
    const size_t nq = n * D.Q, nkq = nq * K;
    MQ_CUDA(cudaMalloc((void**)&D.ref, nq * sizeof(double)));
    MQ_CUDA(cudaMalloc((void**)&D.sum, nkq * sizeof(double)));
    MQ_CUDA(cudaMalloc((void**)&D.sumsq, nkq * sizeof(double)));
    MQ_CUDA(cudaMalloc((void**)&D.n_models, n * sizeof(int64_t)));
    MQ_CUDA(cudaMalloc((void**)&D.batch_len, n * sizeof(int32_t)));
    MQ_CUDA(cudaMalloc((void**)&D.full_batches, n * sizeof(int32_t)));
    cudaStream_t st = h->stream;
    MQ_CUDA(cudaMemsetAsync(D.ref, 0, nq * sizeof(double), st));
    MQ_CUDA(cudaMemsetAsync(D.sum, 0, nkq * sizeof(double), st));
    MQ_CUDA(cudaMemsetAsync(D.sumsq, 0, nkq * sizeof(double), st));
    MQ_CUDA(cudaMemsetAsync(D.n_models, 0, n * sizeof(int64_t), st));
    MQ_CUDA(cudaMemsetAsync(D.full_batches, 0, n * sizeof(int32_t), st));
    {
        std::vector<int32_t> one(n, 1);   // every chain starts with batches of one model
        MQ_CUDA(cudaMemcpyAsync(D.batch_len, one.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        MQ_CUDA(cudaStreamSynchronize(st));
    }
    D.on = 1;
    return MQ_OK;
}

void diag_destroy(Handle* h)
{
    Diag& D = h->diag;
    if (D.ref || D.scratch) {
        cudaSetDevice(h->device);
        if (h->stream) cudaStreamSynchronize(h->stream);
    }
    cudaFree(D.ref); cudaFree(D.sum); cudaFree(D.sumsq); cudaFree(D.n_models); cudaFree(D.batch_len); cudaFree(D.full_batches);
    cudaFree(D.scratch);
    memset(&D, 0, sizeof D);
}

}  // namespace mq

using namespace mq;

extern "C" int mq_diag_begin(mq_handle* hh, int64_t burn_in, int n_batches, mq_diag_dims* dims)
{
    if (!hh) { set_error("mq_diag_begin: null"); return MQ_ERR_ARG; }
    if (burn_in < 0 || n_batches < 8 || n_batches > 64 || (n_batches & 1)) {
        set_error("mq_diag_begin: burn_in %lld, n_batches %d (burn_in >= 0; n_batches even, 8 .. 64)", (long long)burn_in, n_batches);
        return MQ_ERR_ARG;
    }
    Handle* h = &hh->h;
    MQ_CUDA(cudaSetDevice(h->device));
    const int rc = diag_alloc(h, n_batches, (long long)burn_in);
    if (rc != MQ_OK) { diag_destroy(h); return rc; }
    if (dims) { dims->n_quantities = h->diag.Q; dims->nz = h->nz; dims->n_events = h->ne; dims->n_stations = h->ns; dims->n_batches = n_batches; }
    return MQ_OK;
}

extern "C" int mq_diag_chains(mq_handle* hh, double* ref, double* sum, double* sumsq, int32_t* batch_len, int32_t* full_batches,
                              int64_t* n_models)
{
    if (!hh) { set_error("mq_diag_chains: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    const Diag& D = h->diag;
    if (!D.on) { set_error("mq_diag_chains: mq_diag_begin was not called"); return MQ_ERR_STATE; }
    MQ_CUDA(cudaSetDevice(h->device));
    int rc = flags_poll(h, true);
    if (rc != MQ_OK) return rc;
    cudaStream_t s = h->stream;
    const size_t n = h->n, nq = n * D.Q, nkq = nq * D.K;
#define GET(dst, src, cnt) if (dst) MQ_CUDA(cudaMemcpyAsync(dst, src, (cnt) * sizeof(*(dst)), cudaMemcpyDeviceToHost, s))
    GET(ref, D.ref, nq); GET(sum, D.sum, nkq); GET(sumsq, D.sumsq, nkq);
    GET(batch_len, D.batch_len, n); GET(full_batches, D.full_batches, n); GET(n_models, D.n_models, n);
#undef GET
    MQ_CUDA(cudaStreamSynchronize(s));
    return check_device_errors(h);
}

extern "C" int mq_diag_summary(mq_handle* hh, int collective, double* mean, double* sd, double* rhat, double* ess, int64_t* n_models,
                               int32_t* chains_used)
{
    if (!hh) { set_error("mq_diag_summary: null"); return MQ_ERR_ARG; }
    Handle* h = &hh->h;
    Diag& D = h->diag;
    MQ_CUDA(cudaSetDevice(h->device));
    int rc = flags_poll(h, true);     // an error of an earlier asynchronous call comes first
    if (rc != MQ_OK) return rc;
    if (!D.on) { set_error("mq_diag_summary: mq_diag_begin was not called"); return MQ_ERR_STATE; }
    const int Q = D.Q, n = h->n;
    const DiagPlan P = diag_plan(n, Q);
    if (D.scratch_bytes < P.doubles * sizeof(double)) {
        cudaFree(D.scratch);
        D.scratch = nullptr; D.scratch_bytes = 0;
        MQ_CUDA(cudaMalloc((void**)&D.scratch, P.doubles * sizeof(double)));
        D.scratch_bytes = P.doubles * sizeof(double);
    }
    double* w = D.scratch;
    cudaStream_t st = h->stream;
    const dim3 grid_g(P.xb, P.groups), grid_q(P.xb);
    diag_chains_kernel<<<grid_g, kDiagThreads, 0, st>>>(D, n, P.per_group, w + P.part, w + P.mu);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    diag_combine_kernel<<<grid_q, kDiagThreads, 0, st>>>(w + P.part, P.groups, kParts, Q, w + P.tot1);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    if (collective) { rc = comm_allreduce_sum(h, w + P.tot1, kParts * (size_t)Q); if (rc != MQ_OK) return rc; }
    diag_spread_kernel<<<grid_g, kDiagThreads, 0, st>>>(D, n, P.per_group, w + P.tot1, w + P.mu, w + P.part2);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    diag_combine_kernel<<<grid_q, kDiagThreads, 0, st>>>(w + P.part2, P.groups, 1, Q, w + P.tot2);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    if (collective) { rc = comm_allreduce_sum(h, w + P.tot2, (size_t)Q); if (rc != MQ_OK) return rc; }
    diag_final_kernel<<<grid_q, kDiagThreads, 0, st>>>(Q, w + P.tot1, w + P.tot2, w + P.out);
    count_launch();
    MQ_CUDA(cudaGetLastError());
    double counts[2] = {0.0, 0.0};   // chains used and N, the same for every quantity: those of quantity 0
    const double* out = w + P.out;
    if (mean) MQ_CUDA(cudaMemcpyAsync(mean, out, Q * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (sd) MQ_CUDA(cudaMemcpyAsync(sd, out + Q, Q * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (rhat) MQ_CUDA(cudaMemcpyAsync(rhat, out + 2 * (size_t)Q, Q * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (ess) MQ_CUDA(cudaMemcpyAsync(ess, out + 3 * (size_t)Q, Q * sizeof(double), cudaMemcpyDeviceToHost, st));
    MQ_CUDA(cudaMemcpyAsync(&counts[0], w + P.tot1, sizeof(double), cudaMemcpyDeviceToHost, st));
    MQ_CUDA(cudaMemcpyAsync(&counts[1], w + P.tot1 + 6 * (size_t)Q, sizeof(double), cudaMemcpyDeviceToHost, st));
    MQ_CUDA(cudaStreamSynchronize(st));
    if (chains_used) *chains_used = (int32_t)(counts[0] + 0.5);
    if (n_models) *n_models = (int64_t)(counts[1] + 0.5);
    return check_device_errors(h);
}
