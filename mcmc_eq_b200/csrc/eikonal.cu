// eikonal.cu -- batched Podvin-Lecomte eikonal kernels for sm_100a.
//
// Replaces the nz serial calls of time_2d() per phase and chain in the reference
// (src/misfit.c:270-289 -> src/time_2d.c:301) by one launch over every
// (chain, phase, source depth) triple.  One lane owns one solve: the update order of
// the expanding-box scheme is sequential inside a solve and must be kept for parity
// (SURVEY.md section 7 H1), so the parallelism is across solves.
#include "eikonal.cuh"
#include "eik_core.cuh"
#include "eik_fast.cuh"
#include "eik_march.cuh"
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include "launch_count.h"
#include <cub/device/device_radix_sort.cuh>

namespace mq {

constexpr float kInfM = eik::kInf;
constexpr int kFineNodes = 22 * 43;   // refined grid of a left-edge source, src/time_2d.c:844-864

// What the fused, fine and pipelined kernels read of the work space (EikWork; the generic kernel takes the window alone:
// given the whole view its stack frame grows).  The order is set only when it was filled for the batch.
struct EikView {
    float* window;
    float* slices;
    const int32_t* order;
    int32_t* task_counter;
    float* tie;
    int pipe_slices;
};

// Solves per item of a table-mode batch: one per depth (parity) or one per receiver row (reciprocal).
__host__ __device__ inline int eik_sources(const EikBatch& b) { return b.src_rows ? b.n_src_rows : b.nz; }

// Floats of a per-warp window of the generic kernel (time field + refined grid, lane-interleaved): EikWork::window holds
// EikWork::warps of them.  The other kernels need less per warp and take as many warps as fit (warps_fitting).
static size_t eik_scratch_floats_per_warp(int nxmod, int nz)
{
    return ((size_t)nxmod * nz + kFineNodes) * 32;
}

// Solve g of a batch: its source depth, its slowness column (item), where its output starts in the item's table and the
// stride between its output rows (b.rows[r] goes to out_off + r*out_rstride).  Table mode decodes g as parity or, with
// src_rows, reciprocal tables (EikBatch::src_rows); list mode takes src_iz[g] and column g.
struct TableSolve {
    int iz, item;
    size_t out_off;
    long out_rstride;
};
__device__ __forceinline__ TableSolve table_solve(const EikBatch& b, int n_items, int g)
{
    TableSolve t;
    if (b.src_iz) {
        t.iz = b.src_iz[g];
        t.item = g;
        t.out_off = (size_t)t.iz * b.xpitch;
        t.out_rstride = (long)b.nz * b.xpitch;
    } else if (b.src_rows) {
        const int rho = g / n_items;
        t.item = g - rho * n_items;
        t.iz = b.src_rows[rho];
        t.out_off = (size_t)rho * b.n_rows * b.xpitch;
        t.out_rstride = b.xpitch;
    } else {
        t.iz = g / n_items;
        t.item = g - t.iz * n_items;
        t.out_off = (size_t)t.iz * b.xpitch;
        t.out_rstride = (long)b.nz * b.xpitch;
    }
    return t;
}

// Generic kernel: the whole time field of a lane lives in global memory, interleaved by
// lane (node i of lane l at scratch[i*32 + l]) so that lanes that sweep the same node
// -- the common case, all lanes of a warp share the source depth -- touch one 128-byte line.
__global__ void __launch_bounds__(128)
eik_generic_kernel(EikBatch b, float* window)
{
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int warp = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int n_warps = gridDim.x * warps_per_block;
    const int nodes = b.nxmod * b.nz;
    float* W = window + (size_t)warp * (((size_t)nodes + kFineNodes) * 32) + lane;
    float* WF = W + (size_t)nodes * 32;
    const int n_items = b.n_items_dev ? *b.n_items_dev : b.n_items;
    const int n_solves = b.src_iz ? b.n_solves : n_items * eik_sources(b);
    const int n_tasks = (n_solves + 31) >> 5;

    for (int task = warp; task < n_tasks; task += n_warps) {
        const int g = task * 32 + lane;
        if (g < n_solves) {
            const TableSolve ts = table_solve(b, n_items, g);
            const int iz = ts.iz, item = ts.item;
            const float* s = b.slow + (size_t)item * b.nz;
            const int rc = eik::solve(s, 1, b.nxmod, b.nz, iz, W, WF, 32, nullptr);
            if (b.status) b.status[g] = rc;
            if (b.status_min && rc < 0) atomicMin(b.status_min, rc);
            if (b.full_out) {
                float* o = b.full_out + (size_t)g * nodes;
                for (int i = 0; i < nodes; i++) o[i] = W[(size_t)i * 32];
            }
            if (b.n_rows > 0 && (b.row_out || b.row_out_base)) {
                float* tab = (b.row_out ? b.row_out[item] : b.row_out_base + (size_t)item * b.row_item_stride) + ts.out_off;
                for (int r = 0; r < b.n_rows; r++) {
                    const int j = b.rows[r];
                    float* o = tab + (long)r * ts.out_rstride;
                    for (int x = 0; x < b.nxmod; x++) o[x] = W[((size_t)x * b.nz + j) * 32];
                }
            }
        }
        __syncwarp();
    }
}

// Warps with windows of floats_per_warp floats that fit the work space's window.
static long warps_fitting(const EikWork& w, size_t floats_per_warp)
{
    return (long)((size_t)w.warps * eik_scratch_floats_per_warp(w.nxmod, w.nz) / floats_per_warp);
}

static cudaError_t eik_launch_generic(const EikBatch& b, const EikWork& w, const EikView& v, int n_solves, cudaStream_t stream)
{
    const int n_tasks = (n_solves + 31) / 32;
    const long fit = warps_fitting(w, eik_scratch_floats_per_warp(b.nxmod, b.nz));
    const int warps = n_tasks < fit ? n_tasks : (int)fit;
    const int wpb = 4;
    const int blocks = (warps + wpb - 1) / wpb;
    eik_generic_kernel<<<blocks, wpb * 32, 0, stream>>>(b, v.window);
    count_launch();
    return cudaGetLastError();
}


// ---- warp-synchronous kernel ---------------------------------------------------------------------------
static eikf::Dims fast_dims(int nxmod, int nz)
{
    static int row_march = -1;
    if (row_march < 0) {
        const char* e = getenv("MCMCEQ_ROW_MARCH");
        row_march = (e && e[0] == '0') ? 0 : 1;      // lock-step row sweeps (eik_fast.cuh: row_march), on unless MCMCEQ_ROW_MARCH=0
    }
    eikf::Dims D = eikf::make_dims(nxmod, nz);
    D.row_march = row_march;
    return D;
}
static size_t fast_smem_floats_per_warp(const eikf::Dims& D) { return (size_t)eikf::smem_floats_per_lane(D) * 32; }
static size_t fast_scratch_floats_per_warp(const eikf::Dims& D) { return ((size_t)D.wx * D.nz + kFineNodes) * 32; }

static bool eik_fast_supported(int nxmod, int nz)
{
    if (nxmod < 2 || nz < 2) return false;
    const eikf::Dims D = fast_dims(nxmod, nz);
    return fast_smem_floats_per_warp(D) * sizeof(float) <= 200 * 1024;
}

// One warp per block: a warp owns 32 solves and its slice of shared memory, nothing is shared between warps.
// GLOBAL_SLICE (eik_fine_kernel): planes whose perimeter does not fit shared memory (the 0.1 km fine grid: 2001 depth nodes,
// 6010 floats per lane) keep the same three arrays in a per-warp slice of GLOBAL memory, lane-interleaved like the
// shared-memory slice, so that the lock-step sweeps (rows, the march) touch one 128-byte line per access.  Same code,
// same results; what hides the memory latency is the number of resident warps.
template <bool GLOBAL_SLICE>
__device__ __forceinline__ void eik_fast_body(const EikBatch& b, const EikView& wk, const eikf::Dims& D, float* slice, int lpt)
{
    const int lane = threadIdx.x;
    const int nodes = b.nxmod * b.nz;
    eikf::Lane L;
    if (GLOBAL_SLICE) eikf::carve_global(slice + lane, D, &L);
    else eikf::carve_shared(slice + lane, D, &L);
    L.W = wk.window + (size_t)blockIdx.x * (((size_t)D.wx * D.nz + kFineNodes) * 32) + lane;
    L.WF = L.W + (size_t)D.wx * D.nz * 32;
    const int n_items = b.n_items_dev ? *b.n_items_dev : b.n_items;
    const int n_solves = b.src_iz ? b.n_solves : n_items * eik_sources(b);
    const int n_tasks = (n_solves + lpt - 1) / lpt;

    for (int task = blockIdx.x; task < n_tasks; task += gridDim.x) {
        int g = task * lpt + lane;
        if (lane >= lpt) g = -1;
        else if (wk.order) g = wk.order[g];
        eikf::LaneTask t;
        t.valid = g >= 0 && g < n_solves;
        t.iz = 0; t.slow = nullptr; t.out = nullptr; t.out_rstride = 0; t.full = nullptr; t.hand_col = nullptr; t.hand_x1 = nullptr;
        if (t.valid) {
            const TableSolve ts = table_solve(b, n_items, g);
            t.iz = ts.iz;
            const int item = ts.item;
            t.slow = b.slow + (size_t)item * b.nz;
            if (b.n_rows > 0 && (b.row_out || b.row_out_base)) {
                float* tab = b.row_out ? b.row_out[item] : b.row_out_base + (size_t)item * b.row_item_stride;
                t.out = tab + ts.out_off;
                t.out_rstride = ts.out_rstride;
            }
            if (b.full_out) t.full = b.full_out + (size_t)g * nodes;
        }
        const int rc = eikf::solve_warp<GLOBAL_SLICE>(D, L, t, b.rows, b.n_rows);
        if (t.valid) {
            if (b.status) b.status[g] = rc;
            if (b.status_min && rc < 0) atomicMin(b.status_min, rc);
        }
        __syncwarp();
    }
}

// lanes_per_task: lanes of a warp that carry a solve (32, 16, 8 or 4)
__global__ void __launch_bounds__(32, 9) eik_fast_kernel(EikBatch b, EikView wk, eikf::Dims D, int lanes_per_task)
{
    extern __shared__ float smem[];
    eik_fast_body<false>(b, wk, D, smem, lanes_per_task);
}

__global__ void __launch_bounds__(32, 8) eik_fine_kernel(EikBatch b, EikView wk, eikf::Dims D, int lanes_per_task)
{
    eik_fast_body<true>(b, wk, D, wk.slices + (size_t)blockIdx.x * ((size_t)eikf::gmem_floats_per_lane(D) * 32), lanes_per_task);
}

// ---- regrouping of solves --------------------------------------------------------------------------------------
// What a solve does before its march is decided by the layering round its source: the half-width of the
// quasi-homogeneous box (distance to the nearest interface above and below, src/time_2d.c:598-644) selects the kind
// of initialisation and the size of the seed box, the next interfaces decide when rows start to carry head waves.
// Key = source depth (major, so that the lanes of a warp share the box schedule; in ascending order: measured better than edges-first or middle-first), then
// those distances.
__global__ void eik_key_kernel(EikBatch b, int max_solves, uint64_t* keys, int32_t* vals)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= max_solves) return;
    const int n_items = b.n_items_dev ? *b.n_items_dev : b.n_items;
    const int n_solves = n_items * eik_sources(b);
    if (g >= n_solves) { keys[g] = ~0ull; vals[g] = -1; return; }
    const TableSolve ts = table_solve(b, n_items, g);
    const int iz = ts.iz, item = ts.item;
    const float* s = b.slow + (size_t)item * b.nz;
    const int my = b.nz - 1;
    const int ysc = (iz == my) ? iz - 1 : iz;
    const float hs0 = s[ysc], tol = hs0 * 0.001f;
    // run lengths of the layering seen from the source cell: three layers below and above, 5 bits each
    // (thickness in cells capped at 15, and whether the next layer is faster); 31 = the model ends there
    auto runs = [&](int dir, int last, uint64_t* f) {
        int y = ysc;
        float ref = hs0;
        bool ended = false;
        for (int layer = 0; layer < 3; layer++) {
            if (ended) { f[layer] = 31; continue; }
            int len = 0;
            while (y != last && fabsf(s[y + dir] - ref) <= tol) { y += dir; if (len < 15) len++; }
            if (y == last) { f[layer] = 31; ended = true; continue; }
            const int faster = s[y + dir] < ref;
            ref = s[y + dir];
            y += dir;
            f[layer] = (uint64_t)(len << 1 | faster);
        }
    };
    uint64_t dn[3], up[3];
    runs(+1, my - 1, dn);
    runs(-1, 0, up);
    const uint64_t d0 = dn[0], d1 = dn[1], d2 = dn[2], u0 = up[0], u1 = up[1], u2 = up[2];
    // half-width of the seed box first: it decides the kind of initialisation (src/time_2d.c:682-711)
    const uint64_t wd = (d0 == 31) ? 15 : (d0 >> 1), wu = (u0 == 31) ? 15 : (u0 >> 1), w = wd < wu ? wd : wu;
    (void)u2;
    keys[g] = ((uint64_t)iz << 32) | (w << 28) | (d0 << 23) | (u0 << 18) | (d1 << 13) | (u1 << 8) | (d2 << 3);
    vals[g] = g;
}

// Bytes of the sort buffers (EikWork::sort) for up to max_solves solves.
static size_t eik_order_bytes(int max_solves)
{
    const size_t n = ((size_t)max_solves + 31) / 32 * 32;
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const int32_t*)nullptr,
                                    (int32_t*)nullptr, (int)n, 0, 44);
    return 2 * n * sizeof(uint64_t) + n * sizeof(int32_t) + ((tmp + 255) / 256 * 256) + 1024;
}

// Fills wk.order[0 .. round_up(max_solves, 32)): order[j] = the solve g (source * n_items + item) that lane j % 32 of warp
// task j / 32 runs, or -1.
static cudaError_t eik_order_tasks(const EikBatch& b, const EikWork& wk, cudaStream_t stream)
{
    const int max_solves = b.n_items * eik_sources(b);
    if (max_solves <= 0) return cudaSuccess;
    const size_t n = ((size_t)max_solves + 31) / 32 * 32;
    char* w = (char*)wk.sort;
    uint64_t* k_in = (uint64_t*)w;               w += n * sizeof(uint64_t);
    uint64_t* k_out = (uint64_t*)w;              w += n * sizeof(uint64_t);
    int32_t* v_in = (int32_t*)w;                 w += n * sizeof(int32_t);
    w = (char*)(((uintptr_t)w + 255) / 256 * 256);
    size_t tmp = wk.sort_bytes - (size_t)(w - (char*)wk.sort);
    eik_key_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(b, (int)n, k_in, v_in);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    // source depth needs at most 12 bits above bit 32 (nz <= 4096)
    e = cub::DeviceRadixSort::SortPairs(w, tmp, k_in, k_out, v_in, wk.order, (int)n, 0, 44, stream);
    count_launch(3);
    return e;
}

// ---- the pipelined kernel: box phase in shared memory, march in tensor memory, in ONE persistent CTA per SM --------------
// The fused kernel holds 9 warps per SM because every warp keeps 24.7 KB of shared memory for its whole life, although it
// only needs it for the box phase (per-lane indices); the march (warp-uniform indices) can live in TMEM.  Here 12 warps
// per SM share the shared-memory slices (7 with the second column buffer of the lock-step box phase, Dims::lock_cols) and 8 TMEM sets (past column, current column, slowness column = 3 x 64
// columns; two sets per lane quarter): a warp takes a slice for the box phase of a task, moves the task's last column and
// slowness column into a TMEM set, gives the slice back and marches in tensor memory.  At any time about half of the warps
// are in the latency-bound box phase and half in the issue-bound march, and there are 12 of them instead of 9 (168 registers each, the most 12 warps allow: no spills, no stack frame;
// tests/test_sass_footprint_cpu.py).
// Resources are taken in a fixed order (slice, then TMEM set; the tie scratch last and never while waiting for anything
// else), holders of a TMEM set never wait for a slice: no cycle, no deadlock.
// Two instantiations, chosen by the depth of the plane (pipe_shape): column arrays of CA = 64 nodes for nz <= 62 (the Example
// plane), and CA = 128 for 88 <= nz <= 126, which holds the planes of the example grids refined by halving the spacing.  A CA = 128 set is 384
// columns, so a lane quarter holds one and 4 marches are in flight per SM; slices are 48 - 64 KB at those depths (3 - 4 per
// SM), so fewer warps per CTA (profiles/README.md, deep planes).
constexpr int kPipeWarps = 12;       // CA = 64.  Measured 10 .. 20: 12 - 13 are best at 1024 chains, 12 - 16 equal at 8192 (profiles/README.md)
constexpr int kPipeWarpsDeep = 8;    // CA = 128.  Measured 6, 8, 12: 8 is best or level (profiles/README.md)
constexpr int kPipeMaxCtas = 256;    // one CTA per SM; the tie scratch is sized for this many
// two time columns + slowness column of the tie scratch of a CTA
template <int CA>
constexpr size_t kPipeTieFloats = (size_t)(3 * CA + 2) * 32;
// The instantiation a plane of nz depth nodes takes (ca = 0: none) and its warps per CTA.
struct PipeShape {
    int ca, warps;
};
// Lowest nz for CA = 128: a shallower plane fills too little of the column arrays, and the fused kernel is faster (B200,
// 1024 chains: 21.3 against 22.7 ms per launch at nz = 80, 33.4 against 27.5 at nz = 88; DESIGN.md section 3).
constexpr int kPipeDeepMinNz = 88;
static PipeShape pipe_shape(int nz)
{
    if (nz + 2 <= 64) return {64, kPipeWarps};
    if (nz >= kPipeDeepMinNz && nz + 2 <= 128) return {128, kPipeWarpsDeep};
    return {0, 0};
}

// The box phase of a task.  Until round 2 it had to be compiled as a function of its own: inlined next to the tensor-memory
// march, nvcc 12.9 produced a kernel whose box-region output was wrong (bisected on the GPU in round 1: any variant with the
// call inlined and the top-row site of run_grid present failed).  Printing one solve's box phase from both kernels
// (profiles/README.md r2c) showed what goes wrong: at that site the row's own strip slowness c came out as the far side's c2.
// With the two reads volatile (eik_fast.cuh, run_grid) the inlined kernel is bit-identical to the fused one and 8 % faster
// (LDS / STS instead of generic loads and stores); tests/test_pipe_gpu.py compares the two kernels bit for bit on four model
// families and guards this.  The columns of the growing box are swept in lock-step (Dims::lock_cols).
// Arguments by value: as references they would live in the caller's stack frame and be re-read through it.
// x1 receives the column at which the box phase ended (-1: nothing left to march).
__device__ __forceinline__ int solve_warp_call(eikf::Dims D, eikf::Lane L, eikf::LaneTask t, const int* rows, int n_rows, int* x1_out)
{
    int x1 = -1;
    t.hand_x1 = &x1;
    const int rc = eikf::solve_warp<false, true>(D, L, t, rows, n_rows);
    *x1_out = x1;
    return rc;
}

struct PipeCtl {
    uint32_t tmem;                   // base address of the CTA's 512 TMEM columns
    unsigned slice_free;             // bit i: shared-memory slice i is free
    unsigned tset_free[4];           // per lane quarter: bit i: TMEM set i is free
    int tie_lock;
};

__device__ __forceinline__ int pipe_acquire(unsigned* mask, int lane)
{
    int got = -1;
    if (lane == 0) {
        for (;;) {
            const unsigned m = *(volatile unsigned*)mask;
            if (m) {
                const int bit = __ffs(m) - 1;
                if (atomicAnd(mask, ~(1u << bit)) & (1u << bit)) { got = bit; break; }
            } else {
                __nanosleep(20000);
            }
        }
        __threadfence_block();
    }
    return __shfl_sync(0xffffffffu, got, 0);
}
__device__ __forceinline__ void pipe_release(unsigned* mask, int bit, int lane)
{
    __syncwarp();
    if (lane == 0) { __threadfence_block(); atomicOr(mask, 1u << bit); }
}

// CA: nodes -1 .. CA-2 per TMEM column array (nz <= CA - 2); WARPS: warps per CTA; RECIP: reciprocal tables
// (EikBatch::src_rows, with rows = 0 .. nz-1): every row of each column is output.
template <int CA, int WARPS, bool RECIP>
__device__ __forceinline__ void eik_pipe_body(const EikBatch& b, const EikView& wk, const eikf::Dims& D)
{
    constexpr int NB = CA / 4;
    constexpr int kSets = 512 / (3 * CA);        // TMEM sets per lane quarter: 2 at CA = 64, 1 at CA = 128
    extern __shared__ float smem_p[];
    __shared__ PipeCtl ctl;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, quarter = warp & 3;
    if (warp == 0) eikm::tmem_alloc<512>(&ctl.tmem);
    if (threadIdx.x == 0) {
        ctl.slice_free = (1u << wk.pipe_slices) - 1u;
        for (int q = 0; q < 4; q++) ctl.tset_free[q] = (1u << kSets) - 1u;
        ctl.tie_lock = 0;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const size_t slice_floats = (size_t)eikf::smem_floats_per_lane(D) * 32;
    // scratch of the literal walk for a column with an exact tie (4 in 100 000): global memory, one per CTA, under a lock
    float* tieP = wk.tie + (size_t)blockIdx.x * kPipeTieFloats<CA> + 32 + lane;   // node k at tieP[k*32], k = -1 .. CA-2
    float* tieC = tieP + (size_t)CA * 32;
    float* tieS = tieC + (size_t)CA * 32 + 32;                             // cell k at tieS[k*32], k = -2 .. CA-1
    const int nz = b.nz, ke = nz - 1, mx = b.nxmod - 1;
    const int n_items = b.n_items_dev ? *b.n_items_dev : b.n_items;
    const int n_solves = n_items * (RECIP ? b.n_src_rows : nz);
    const int n_tasks = (n_solves + 31) >> 5;
    const size_t wfloats = ((size_t)D.wx * D.nz + kFineNodes) * 32;
    float* Wbase = wk.window + (size_t)(blockIdx.x * WARPS + warp) * wfloats + lane;

    for (;;) {
        int task = 0;
        if (lane == 0) task = atomicAdd(wk.task_counter, 1);
        task = __shfl_sync(0xffffffffu, task, 0);
        if (task >= n_tasks) break;
        int g = task * 32 + lane;
        if (wk.order) g = wk.order[g];
        // ---- box phase on a shared-memory slice
        const int sl = pipe_acquire(&ctl.slice_free, lane);
        eikf::Lane L;
        eikf::carve_shared(smem_p + (size_t)sl * slice_floats + lane, D, &L);
        L.W = Wbase;
        L.WF = L.W + (size_t)D.wx * D.nz * 32;
        eikf::LaneTask t;
        t.valid = g >= 0 && g < n_solves;
        t.iz = 0; t.slow = nullptr; t.out = nullptr; t.out_rstride = 0; t.full = nullptr;
        int x1 = -1;
        t.hand_col = L.COL;          // the last column of the box phase already sits there
        t.hand_x1 = nullptr;         // set inside solve_warp_call
        if (t.valid) {
            // table_solve with the mode known at compile time (no list mode here)
            const int s = g / n_items, item = g - s * n_items;
            t.iz = RECIP ? b.src_rows[s] : s;
            t.slow = b.slow + (size_t)item * nz;
            float* tab = b.row_out ? b.row_out[item] : b.row_out_base + (size_t)item * b.row_item_stride;
            t.out = tab + (RECIP ? (size_t)s * nz * b.xpitch : (size_t)s * b.xpitch);
            t.out_rstride = RECIP ? (long)b.xpitch : (long)nz * b.xpitch;
        }
        const int rc = solve_warp_call(D, L, t, b.rows, b.n_rows, &x1);
        if (t.valid && b.status_min && rc < 0) atomicMin(b.status_min, rc);
        const bool live = x1 >= 0 && x1 < mx;
        if (!__any_sync(0xffffffffu, live)) { pipe_release(&ctl.slice_free, sl, lane); continue; }
        // ---- move the task into a TMEM set of this warp's lane quarter, give the slice back
        const int ts = pipe_acquire(&ctl.tset_free[quarter], lane);
        // set ts of the quarter: columns [3 CA ts, 3 CA (ts + 1)) = past | current | slowness.  Columns [3 CA kSets, 512) stay
        // unused (at CA = 64: a third set with its slowness column in shared memory costs two slices and was slower,
        // profiles/README.md)
        const uint32_t tset = ctl.tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(ts * 3 * CA);
        const uint32_t tS = tset + 2 * CA;
        for (int q = 0; q < NB; q++) {
            float v[4], w[4];
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int k = 4 * q - 1 + c;
                v[c] = (k >= 0 && k <= ke) ? (live ? L.COL[(size_t)k * 32] : 0.f) : eikm::sentinel(k, ke);
                w[c] = (live && k >= 0 && k < ke) ? L.S[(size_t)k * 32] : kInfM;
            }
            eikm::tmem_st4(tset + 4 * q, v);
            eikm::tmem_st4(tS + 4 * q, w);
        }
        eikm::tmem_wait_st();
        pipe_release(&ctl.slice_free, sl, lane);
        // ---- march in tensor memory
        uint32_t tp = tset, tc = tset + CA;
        const int xlo = __reduce_min_sync(0xffffffffu, live ? x1 : 0x7fffffff);
        const int xhi = __reduce_max_sync(0xffffffffu, live ? x1 : -1);
        for (int line = xlo + 1; line <= mx; line++) {
            const bool need = live && line > x1;
            const bool tie = (line <= xhi) ? eikm::tmem_sweep<NB, true>(need, tp, tc, tS)
                                           : eikm::tmem_sweep<NB, false>(need, tp, tc, tS);
            eikm::tmem_wait_st();
            if (__any_sync(0xffffffffu, tie)) {
                // an exact tie in the past column: the literal walk (march_sweep) on a shared-memory copy, under the CTA's lock
                if (lane == 0) { while (atomicCAS(&ctl.tie_lock, 0, 1) != 0) __nanosleep(500); __threadfence_block(); }
                __syncwarp();
                for (int q = 0; q < NB; q++) {
                    float v[4], w[4];
                    eikm::tmem_ld4(tp + 4 * q, v);
                    eikm::tmem_ld4(tS + 4 * q, w);
                    eikm::tmem_wait_ld(v, w);
#pragma unroll
                    for (int c = 0; c < 4; c++) { tieP[(long)(4 * q - 1 + c) * 32] = v[c]; tieS[(long)(4 * q - 1 + c) * 32] = w[c]; }
                }
                tieS[-64] = kInfM;
                if (tie) { tieP[-32] = eikf::kStop; tieP[(long)(ke + 1) * 32] = eikf::kStop; }
                int nohint = -1;
                eikf::march_sweep(tie, tieP, tieC, tieS, ke, &nohint);
                for (int q = 0; q < NB; q++) {
                    float v[4];
                    eikm::tmem_ld4(tc + 4 * q, v);
                    eikm::tmem_wait_ld(v);
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        const int k = 4 * q - 1 + c;
                        if (tie && k >= 0 && k <= ke) v[c] = tieC[(long)k * 32];
                    }
                    eikm::tmem_st4(tc + 4 * q, v);
                }
                eikm::tmem_wait_st();
                __syncwarp();
                if (lane == 0) { __threadfence_block(); atomicExch(&ctl.tie_lock, 0); }
            }
            eikm::tmem_st1(tc, eikf::kEdge);
            if (CA == 64) {
                for (int k = ke + 1; k <= CA - 2; k++) eikm::tmem_st1(tc + k + 1, eikm::sentinel(k, ke));
            } else {
                // up to 64 nodes at CA = 128: single stores up to the next group of four columns, .x4 stores from there
                int k = ke + 1;
                for (; k <= CA - 2 && ((k + 1) & 3); k++) eikm::tmem_st1(tc + k + 1, eikm::sentinel(k, ke));
                for (; k <= CA - 2; k += 4) {
                    const float v[4] = {eikm::sentinel(k, ke), eikm::sentinel(k + 1, ke), eikm::sentinel(k + 2, ke), eikm::sentinel(k + 3, ke)};
                    eikm::tmem_st4(tc + k + 1, v);
                }
            }
            eikm::tmem_wait_st();
            if (RECIP) {
                // every row of the column: .x4 loads of four groups (16 nodes) and one wait per four groups (groups
                // 4q0 .. 4q0+3 never pass group NB-1: NB is a multiple of four)
                const int q_end = (ke + 1) / 4 + 1;      // node ke is in group (ke + 1) / 4
                for (int q0 = 0; q0 < q_end; q0 += 4) {
                    float v[4][4];
#pragma unroll
                    for (int u = 0; u < 4; u++) eikm::tmem_ld4(tc + 4 * (q0 + u), v[u]);
                    eikm::tmem_wait_ld(v);
                    if (need) {
#pragma unroll
                        for (int u = 0; u < 4; u++)
#pragma unroll
                            for (int c = 0; c < 4; c++) {
                                const int k = 4 * (q0 + u) - 1 + c;
                                if (k >= 0 && k <= ke) t.out[(long)k * t.out_rstride + line] = v[u][c];
                            }
                    }
                }
            } else {
                for (int r = 0; r < b.n_rows; r++) {
                    float v = eikm::tmem_ld1(tc + b.rows[r] + 1);
                    eikm::tmem_wait_ld(v);
                    if (need) t.out[(long)r * t.out_rstride + line] = v;
                }
            }
            const uint32_t tt = tp; tp = tc; tc = tt;
        }
        pipe_release(&ctl.tset_free[quarter], ts, lane);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) eikm::tmem_dealloc<512>(ctl.tmem);
}

template <int CA, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 1) eik_pipe_kernel(EikBatch b, EikView wk, eikf::Dims D)
{
    eik_pipe_body<CA, WARPS, false>(b, wk, D);
}
// The reciprocal-table instantiation (a kernel of its own name: the parity kernel's code stays as it is)
template <int CA, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 1) eik_pipe_recip_kernel(EikBatch b, EikView wk, eikf::Dims D)
{
    eik_pipe_body<CA, WARPS, true>(b, wk, D);
}

static bool eik_pipe_enabled()
{
    static int enabled = -1;
    if (enabled < 0) {
        const char* e = getenv("MCMCEQ_EIKONAL_PIPE");
        enabled = (e && e[0] == '0') ? 0 : 1;     // on unless MCMCEQ_EIKONAL_PIPE=0
    }
    return enabled;
}

static eikf::Dims pipe_dims(int nxmod, int nz)
{
    eikf::Dims D = fast_dims(nxmod, nz);
    // Lock-step columns in the box phase (a second column buffer per slice: 7 slices instead of 9 on the Example plane).
    // Kernel ms per launch at 1024 / 2048 / 4096 / 8192 chains with the box phase inlined: 7.70 / 13.99 / 26.42 / 51.07
    // against 8.03 / 14.24 / 26.66 / 51.07 with the per-lane in-place walk (profiles/README.md r2c).
    D.lock_cols = 1;
    return D;
}

static size_t eik_pipe_tie_floats(int nz)
{
    return (size_t)kPipeMaxCtas * (pipe_shape(nz).ca == 128 ? kPipeTieFloats<128> : kPipeTieFloats<64>);
}

static cudaError_t eik_launch_pipe(const EikBatch& b, const EikWork& w, const EikView& v, long fit, int n_solves, cudaStream_t stream)
{
    void (*const kernel)(EikBatch, EikView, eikf::Dims) =
        b.src_rows ? (w.pipe_ca == 64 ? eik_pipe_recip_kernel<64, kPipeWarps> : eik_pipe_recip_kernel<128, kPipeWarpsDeep>)
                   : (w.pipe_ca == 64 ? eik_pipe_kernel<64, kPipeWarps> : eik_pipe_kernel<128, kPipeWarpsDeep>);
    const int n_tasks = (n_solves + 31) / 32;
    int blocks = (n_tasks + w.pipe_warps - 1) / w.pipe_warps;
    if (blocks > w.sms) blocks = w.sms;
    if ((long)blocks * w.pipe_warps > fit) blocks = (int)(fit / w.pipe_warps);
    cudaError_t e = cudaMemsetAsync(w.task_counter, 0, sizeof(int), stream);
    if (e != cudaSuccess) return e;
    kernel<<<blocks, w.pipe_warps * 32, w.pipe_smem, stream>>>(b, v, pipe_dims(b.nxmod, b.nz));
    count_launch();
    return cudaGetLastError();
}

static cudaError_t eik_launch_fast(const EikBatch& b, const EikWork& w, const EikView& v, long fit, int n_solves, cudaStream_t stream)
{
    const eikf::Dims D = fast_dims(b.nxmod, b.nz);
    const size_t smem = fast_smem_floats_per_warp(D) * sizeof(float);
    long warps = fit < w.fast_resident ? fit : w.fast_resident;
    // A launch with fewer warp-tasks than warps that can be resident lasts as long as one task, and a task is the shorter
    // the fewer lanes have to wait for each other in the box phase: spread it over the idle warps.
    int lpt = 32;
    while (lpt > 4 && ((long)n_solves + lpt / 2 - 1) / (lpt / 2) <= warps) lpt /= 2;
    const int n_tasks = (n_solves + lpt - 1) / lpt;
    if (warps > n_tasks) warps = n_tasks;
    if (warps < 1) warps = 1;
    eik_fast_kernel<<<(unsigned)warps, 32, smem, stream>>>(b, v, D, lpt);
    count_launch();
    return cudaGetLastError();
}

const char* eik_kernel_name(int which)
{
    static const char* names[kEikKernels] = {"eik_generic_kernel", "eik_fast_kernel", "eik_pipe_kernel", "eik_fine_kernel"};
    return (which >= 0 && which < kEikKernels) ? names[which] : "?";
}

static size_t eik_fine_slice_floats_per_warp(int nxmod, int nz)
{
    return (size_t)eikf::gmem_floats_per_lane(fast_dims(nxmod, nz)) * 32;
}

static cudaError_t eik_launch_fine(const EikBatch& b, const EikWork& w, const EikView& v, long fit, int n_solves, cudaStream_t stream)
{
    const int n_tasks = (n_solves + 31) / 32;
    // one warp per CTA; the slices exist for w.warps warps
    long warps = fit < w.warps ? fit : w.warps;
    if (warps > n_tasks) warps = n_tasks;
    if (warps < 1) warps = 1;
    eik_fine_kernel<<<(unsigned)warps, 32, 0, stream>>>(b, v, fast_dims(b.nxmod, b.nz), 32);
    count_launch();
    return cudaGetLastError();
}

cudaError_t eik_launch(const EikBatch& b, const EikWork& w, cudaStream_t stream, int* which)
{
    int dummy;
    if (!which) which = &dummy;
    if (b.nxmod != w.nxmod || b.nz != w.nz) return cudaErrorInvalidValue;   // the windows are laid out for the work's plane
    static int force_generic = -1;
    if (force_generic < 0) {
        const char* e = getenv("MCMCEQ_EIKONAL");
        force_generic = (e && strcmp(e, "generic") == 0) ? 1 : 0;
    }
    EikView v = {w.window, w.slices, nullptr, w.task_counter, w.tie, w.pipe_slices};
    if (b.regroup && w.order) {
        const cudaError_t e = eik_order_tasks(b, w, stream);
        if (e != cudaSuccess) return e;
        v.order = w.order;
    }
    const int n_solves = b.src_iz ? b.n_solves : b.n_items * eik_sources(b);   // upper bound when n_items_dev is set
    // warps of the fused, fine and pipelined kernels whose windows fit the work space
    const long fit = warps_fitting(w, fast_scratch_floats_per_warp(fast_dims(b.nxmod, b.nz)));
    if (!force_generic && w.pipe_ca && !b.src_iz && !b.full_out && (!b.src_rows || b.n_rows == b.nz)) {
        // worth it (and the per-warp windows suffice) only when there is work for every warp of every SM
        const long full = (long)w.sms * w.pipe_warps;
        if (fit >= full && (n_solves + 31) / 32 >= full) {
            *which = kEikPipe;
            return eik_launch_pipe(b, w, v, fit, n_solves, stream);
        }
    }
    *which = force_generic ? kEikGeneric : w.fast_resident ? kEikFast : (w.slices && b.nxmod >= 2 && b.nz >= 2) ? kEikFine : kEikGeneric;
    if (n_solves <= 0) return cudaSuccess;
    if (*which == kEikFast) return eik_launch_fast(b, w, v, fit, n_solves, stream);
    if (*which == kEikFine) return eik_launch_fine(b, w, v, fit, n_solves, stream);
    return eik_launch_generic(b, w, v, n_solves, stream);
}

// Dynamic shared memory: the kernels that take it may use all a block can opt in to on the device, with the largest
// carveout.  Set on every allocation (it is the same each time), so a kernel's limit is never lowered under a launch
// that relies on it, whatever plane another work space on the device has.
static cudaError_t opt_in_shared(int smem_optin)
{
    const void* kernels[] = {(const void*)eik_fast_kernel,
                             (const void*)eik_pipe_kernel<64, kPipeWarps>, (const void*)eik_pipe_kernel<128, kPipeWarpsDeep>,
                             (const void*)eik_pipe_recip_kernel<64, kPipeWarps>, (const void*)eik_pipe_recip_kernel<128, kPipeWarpsDeep>};
    for (const void* kernel : kernels) {
        cudaFuncAttributes a;
        cudaError_t e = cudaFuncGetAttributes(&a, kernel);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_optin - (int)a.sharedSizeBytes);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t eik_work_alloc(EikWork* w, int nxmod, int nz, int max_solves, bool tables, int device)
{
    *w = EikWork{};
    w->nxmod = nxmod;
    w->nz = nz;
    int smem_optin = 0;
    cudaError_t e = cudaDeviceGetAttribute(&w->sms, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e == cudaSuccess) e = opt_in_shared(smem_optin);
    if (e != cudaSuccess) return e;
    const bool fast = eik_fast_supported(nxmod, nz);
    if (fast) {
        int per_sm = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, eik_fast_kernel, 32,
                                                          fast_smem_floats_per_warp(fast_dims(nxmod, nz)) * sizeof(float));
        if (e != cudaSuccess) return e;
        w->fast_resident = w->sms * (per_sm < 1 ? 1 : per_sm);
    }
    const PipeShape sh = pipe_shape(nz);
    if (tables && fast && sh.ca && eik_pipe_enabled() && w->sms <= kPipeMaxCtas) {
        const size_t slice = fast_smem_floats_per_warp(pipe_dims(nxmod, nz)) * sizeof(float);
        const int n_slices = std::min<int>((int)(((size_t)smem_optin - 256) / slice), sh.warps);
        if (n_slices >= 2) {
            w->pipe_ca = sh.ca;
            w->pipe_warps = sh.warps;
            w->pipe_slices = n_slices;
            w->pipe_smem = (size_t)n_slices * slice;
        }
    }

    // Windows for one full wave of the solves, never more (the fine kernel: 12 warps per SM, the others 16).  Large planes
    // (the 0.1 km fine-grid case: 565 x 2001 nodes = 145 MB of window + 0.8 MB of slice per warp): never more than 70 %
    // of the device memory that is still free (25 % for planes that fit a shared-memory slice); the kernels loop over the
    // tasks with however many warps they are given.  MCMCEQ_SCRATCH_FRACTION overrides the fraction.
    long warps = std::min<long>(((long)max_solves + 31) / 32, (long)w->sms * (fast ? 16 : 12));
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
        double frac = fast ? 0.25 : 0.7;
        if (const char* s = getenv("MCMCEQ_SCRATCH_FRACTION")) { const double f = atof(s); if (f > 0.0 && f < 0.95) frac = f; }
        const size_t per_warp = (eik_scratch_floats_per_warp(nxmod, nz) + (fast ? 0 : eik_fine_slice_floats_per_warp(nxmod, nz))) * sizeof(float);
        const long by_mem = (long)(((double)free_b * frac) / (double)per_warp);
        warps = std::min<long>(warps, std::max<long>(by_mem, 4));
    }
    w->warps = (int)((warps + 3) / 4 * 4);
    e = cudaMalloc(&w->window, (size_t)w->warps * eik_scratch_floats_per_warp(nxmod, nz) * sizeof(float));
    if (e == cudaSuccess && !fast) e = cudaMalloc(&w->slices, (size_t)w->warps * eik_fine_slice_floats_per_warp(nxmod, nz) * sizeof(float));
    // regrouping (planes that do not fit a shared-memory slice keep the natural order: a chain's P and S solves of one
    // source depth are neighbours there, which is the grouping their long box phases want; measured, tools/fine_probe2.py)
    if (e == cudaSuccess && tables && fast) {
        w->sort_bytes = eik_order_bytes(max_solves);
        e = cudaMalloc(&w->sort, w->sort_bytes);
        if (e == cudaSuccess) e = cudaMalloc((void**)&w->order, (((size_t)max_solves + 31) / 32 * 32) * sizeof(int32_t));
    }
    if (e == cudaSuccess && w->pipe_ca) {
        e = cudaMalloc((void**)&w->task_counter, sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMemset(w->task_counter, 0, sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMalloc((void**)&w->tie, eik_pipe_tie_floats(nz) * sizeof(float));
        if (e == cudaSuccess) e = cudaMemset(w->tie, 0, eik_pipe_tie_floats(nz) * sizeof(float));
    }
    if (e != cudaSuccess) eik_work_free(w);
    return e;
}

void eik_work_free(EikWork* w)
{
    cudaFree(w->window); cudaFree(w->slices); cudaFree(w->sort); cudaFree(w->order); cudaFree(w->task_counter); cudaFree(w->tie);
    *w = EikWork{};
}

}  // namespace mq
