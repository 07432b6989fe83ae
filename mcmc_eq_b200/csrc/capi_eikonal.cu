// capi_eikonal.cu -- C ABI: stand-alone eikonal entry points (mq_time_2d, mq_eikonal_batch).
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <vector>

#include "../../include/mcmceq_b200.h"
#include "eikonal.cuh"
#include "errors.h"
#include "launch_count.h"

namespace mq {
std::atomic<int64_t> g_launches{0};
thread_local char g_err[512] = "";
void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}
}  // namespace mq

using namespace mq;

extern "C" const char* mq_version(void) { return "mcmc_eq_b200 0.1 (sm_100a)"; }
extern "C" const char* mq_last_error(void) { return g_err; }
extern "C" int64_t mq_launch_count(void) { return g_launches.load(); }

extern "C" int mq_eikonal_batch(const float* slow, const int32_t* src_iz, int n, int nxmod, int nz, float* t_out,
                                int32_t* status, int device)
{
    if (!slow || !src_iz || !t_out || n < 0 || nxmod < 2 || nz < 2) {
        set_error("mq_eikonal_batch: bad argument");
        return MQ_ERR_ARG;
    }
    if (n == 0) return MQ_OK;
    for (int i = 0; i < n; i++)
        if (src_iz[i] < 0 || src_iz[i] >= nz) {
            set_error("mq_eikonal_batch: src_iz[%d]=%d outside [0,%d)", i, src_iz[i], nz);
            return MQ_ERR_ARG;
        }
    MQ_CUDA(cudaSetDevice(device));
    const size_t nodes = (size_t)nxmod * nz;
    // bound the device footprint: process the batch in chunks
    const int chunk_max = 32 * 1024;
    float *d_slow = nullptr, *d_out = nullptr;
    int32_t *d_iz = nullptr, *d_st = nullptr;
    EikWork work = {};
    const int chunk = n < chunk_max ? n : chunk_max;
    int rc = MQ_OK;
    cudaError_t e;
#define TRY(x) do { e = (x); if (e != cudaSuccess) { set_error("%s: %s", #x, cudaGetErrorString(e)); rc = MQ_ERR_CUDA; goto done; } } while (0)
    TRY(cudaMalloc(&d_slow, (size_t)chunk * nz * sizeof(float)));
    TRY(cudaMalloc(&d_iz, (size_t)chunk * sizeof(int32_t)));
    TRY(cudaMalloc(&d_st, (size_t)chunk * sizeof(int32_t)));
    TRY(cudaMalloc(&d_out, (size_t)chunk * nodes * sizeof(float)));
    TRY(eik_work_alloc(&work, nxmod, nz, chunk, false, device));
    for (int off = 0; off < n; off += chunk) {
        const int m = (n - off) < chunk ? (n - off) : chunk;
        TRY(cudaMemcpy(d_slow, slow + (size_t)off * nz, (size_t)m * nz * sizeof(float), cudaMemcpyHostToDevice));
        TRY(cudaMemcpy(d_iz, src_iz + off, (size_t)m * sizeof(int32_t), cudaMemcpyHostToDevice));
        EikBatch b = {};
        b.nxmod = nxmod; b.nz = nz; b.slow = d_slow; b.n_items = m; b.src_iz = d_iz; b.n_solves = m;
        b.full_out = d_out; b.status = d_st;
        TRY(eik_launch(b, work, 0));
        TRY(cudaDeviceSynchronize());
        TRY(cudaMemcpy(t_out + (size_t)off * nodes, d_out, (size_t)m * nodes * sizeof(float), cudaMemcpyDeviceToHost));
        std::vector<int32_t> st(m);
        TRY(cudaMemcpy(st.data(), d_st, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToHost));
        for (int i = 0; i < m; i++) {
            if (status) status[off + i] = st[i];
            if (st[i] != 0 && rc == MQ_OK) {
                set_error("mq_eikonal_batch: solve %d returned %d", off + i, st[i]);
                rc = MQ_ERR_SOLVER;
            }
        }
    }
done:
#undef TRY
    cudaFree(d_slow); cudaFree(d_iz); cudaFree(d_st); cudaFree(d_out);
    eik_work_free(&work);
    return rc;
}

extern "C" int mq_time_2d(const float* hs, float* t, int nx, int ny, float xs, float ys, float eps_init, int messages)
{
    (void)messages;
    if (!hs || !t || nx < 2 || ny < 2) { set_error("mq_time_2d: bad argument"); return MQ_ERR_ARG; }
    const int iz = (int)ys;
    if (xs != 0.f || ys != (float)iz || iz < 0 || iz > ny - 1 || eps_init != 0.001f) {
        set_error("mq_time_2d: only xs == 0, integer ys, eps_init == 0.001 are on the hot path (src/misfit.c:278)");
        return MQ_ERR_UNSUPPORTED;
    }
    // the medium must not vary along x (dummy column nx-1 excluded, it is masked anyway)
    for (int x = 1; x < nx - 1; x++)
        if (memcmp(hs + (size_t)x * ny, hs, (size_t)(ny - 1) * sizeof(float)) != 0) {
            set_error("mq_time_2d: hs varies along x (column %d); only depth-only media are on the hot path", x);
            return MQ_ERR_UNSUPPORTED;
        }
    int dev = 0;
    cudaGetDevice(&dev);
    int32_t st = 0, src = iz;
    const int rc = mq_eikonal_batch(hs, &src, 1, nx, ny, t, &st, dev);
    return rc;
}
