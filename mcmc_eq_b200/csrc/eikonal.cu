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
#include "launch_count.h"
#include <cub/device/device_radix_sort.cuh>

namespace mq {

constexpr float kInfM = eik::kInf;

size_t eik_scratch_floats_per_warp(int nxmod, int nz)
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
eik_generic_kernel(EikBatch b)
{
    const int lane = threadIdx.x & 31;
    const int warps_per_block = blockDim.x >> 5;
    const int warp = blockIdx.x * warps_per_block + (threadIdx.x >> 5);
    const int n_warps = gridDim.x * warps_per_block;
    const int nodes = b.nxmod * b.nz;
    float* W = b.scratch + (size_t)warp * (((size_t)nodes + kFineNodes) * 32) + lane;
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

cudaError_t eik_launch_generic(const EikBatch& b, cudaStream_t stream)
{
    const int n_solves = b.src_iz ? b.n_solves : b.n_items * eik_sources(b);   // upper bound when n_items_dev is set
    if (n_solves <= 0) return cudaSuccess;
    const int n_tasks = (n_solves + 31) / 32;
    const int warps = n_tasks < b.max_warps ? n_tasks : b.max_warps;
    const int wpb = 4;
    const int blocks = (warps + wpb - 1) / wpb;
    eik_generic_kernel<<<blocks, wpb * 32, 0, stream>>>(b);
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

bool eik_fast_supported(int nxmod, int nz)
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
__device__ __forceinline__ void eik_fast_body(const EikBatch& b, const eikf::Dims& D, float* slice, int lpt)
{
    const int lane = threadIdx.x;
    const int nodes = b.nxmod * b.nz;
    eikf::Lane L;
    if (GLOBAL_SLICE) eikf::carve_global(slice + lane, D, &L);
    else eikf::carve_shared(slice + lane, D, &L);
    L.W = b.scratch + (size_t)blockIdx.x * (((size_t)D.wx * D.nz + kFineNodes) * 32) + lane;
    L.WF = L.W + (size_t)D.wx * D.nz * 32;
    const int n_items = b.n_items_dev ? *b.n_items_dev : b.n_items;
    const int n_solves = b.src_iz ? b.n_solves : n_items * eik_sources(b);
    const int n_tasks = (n_solves + lpt - 1) / lpt;

    for (int task = blockIdx.x; task < n_tasks; task += gridDim.x) {
        int g = task * lpt + lane;
        if (lane >= lpt) g = -1;
        else if (b.order) g = b.order[g];
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
__global__ void __launch_bounds__(32, 9) eik_fast_kernel(EikBatch b, eikf::Dims D, int lanes_per_task)
{
    extern __shared__ float smem[];
    eik_fast_body<false>(b, D, smem, lanes_per_task);
}

__global__ void __launch_bounds__(32, 8) eik_fine_kernel(EikBatch b, eikf::Dims D, int lanes_per_task)
{
    eik_fast_body<true>(b, D, b.slice_scratch + (size_t)blockIdx.x * ((size_t)eikf::gmem_floats_per_lane(D) * 32), lanes_per_task);
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

size_t eik_order_bytes(int max_solves)
{
    const size_t n = ((size_t)max_solves + 31) / 32 * 32;
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const int32_t*)nullptr,
                                    (int32_t*)nullptr, (int)n, 0, 44);
    return 2 * n * sizeof(uint64_t) + n * sizeof(int32_t) + ((tmp + 255) / 256 * 256) + 1024;
}

cudaError_t eik_order_tasks(const EikBatch& b, int32_t* order, void* work, size_t work_bytes, cudaStream_t stream)
{
    const int max_solves = b.n_items * eik_sources(b);
    if (max_solves <= 0) return cudaSuccess;
    const size_t n = ((size_t)max_solves + 31) / 32 * 32;
    char* w = (char*)work;
    uint64_t* k_in = (uint64_t*)w;               w += n * sizeof(uint64_t);
    uint64_t* k_out = (uint64_t*)w;              w += n * sizeof(uint64_t);
    int32_t* v_in = (int32_t*)w;                 w += n * sizeof(int32_t);
    w = (char*)(((uintptr_t)w + 255) / 256 * 256);
    size_t tmp = work_bytes - (size_t)(w - (char*)work);
    eik_key_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(b, (int)n, k_in, v_in);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    // source depth needs at most 12 bits above bit 32 (nz <= 4096)
    e = cub::DeviceRadixSort::SortPairs(w, tmp, k_in, k_out, v_in, order, (int)n, 0, 44, stream);
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
__device__ __forceinline__ void eik_pipe_body(const EikBatch& b, const eikf::Dims& D, int n_slices, int* task_counter)
{
    constexpr int NB = CA / 4;
    constexpr int kSets = 512 / (3 * CA);        // TMEM sets per lane quarter: 2 at CA = 64, 1 at CA = 128
    extern __shared__ float smem_p[];
    __shared__ PipeCtl ctl;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, quarter = warp & 3;
    if (warp == 0) eikm::tmem_alloc<512>(&ctl.tmem);
    if (threadIdx.x == 0) {
        ctl.slice_free = (1u << n_slices) - 1u;
        for (int q = 0; q < 4; q++) ctl.tset_free[q] = (1u << kSets) - 1u;
        ctl.tie_lock = 0;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const size_t slice_floats = (size_t)eikf::smem_floats_per_lane(D) * 32;
    // scratch of the literal walk for a column with an exact tie (4 in 100 000): global memory, one per CTA, under a lock
    float* tieP = b.tie_scratch + (size_t)blockIdx.x * kPipeTieFloats<CA> + 32 + lane;   // node k at tieP[k*32], k = -1 .. CA-2
    float* tieC = tieP + (size_t)CA * 32;
    float* tieS = tieC + (size_t)CA * 32 + 32;                             // cell k at tieS[k*32], k = -2 .. CA-1
    const int nz = b.nz, ke = nz - 1, mx = b.nxmod - 1;
    const int n_items = b.n_items_dev ? *b.n_items_dev : b.n_items;
    const int n_solves = n_items * (RECIP ? b.n_src_rows : nz);
    const int n_tasks = (n_solves + 31) >> 5;
    const size_t wfloats = ((size_t)D.wx * D.nz + kFineNodes) * 32;
    float* Wbase = b.scratch + (size_t)(blockIdx.x * WARPS + warp) * wfloats + lane;

    for (;;) {
        int task = 0;
        if (lane == 0) task = atomicAdd(task_counter, 1);
        task = __shfl_sync(0xffffffffu, task, 0);
        if (task >= n_tasks) break;
        int g = task * 32 + lane;
        if (b.order) g = b.order[g];
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
__global__ void __launch_bounds__(WARPS * 32, 1) eik_pipe_kernel(EikBatch b, eikf::Dims D, int n_slices, int* task_counter)
{
    eik_pipe_body<CA, WARPS, false>(b, D, n_slices, task_counter);
}
// The reciprocal-table instantiation (a kernel of its own name: the parity kernel's code stays as it is)
template <int CA, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 1) eik_pipe_recip_kernel(EikBatch b, eikf::Dims D, int n_slices, int* task_counter)
{
    eik_pipe_body<CA, WARPS, true>(b, D, n_slices, task_counter);
}

bool eik_pipe_supported(int nxmod, int nz)
{
    static int enabled = -1;
    if (enabled < 0) {
        const char* e = getenv("MCMCEQ_EIKONAL_PIPE");
        enabled = (e && e[0] == '0') ? 0 : 1;     // on unless MCMCEQ_EIKONAL_PIPE=0
    }
    return enabled && eik_fast_supported(nxmod, nz) && pipe_shape(nz).ca > 0;
}

cudaError_t eik_launch_pipe(const EikBatch& b, int* task_counter, cudaStream_t stream)
{
    if (b.src_iz || b.full_out || !task_counter || !b.tie_scratch) return cudaErrorInvalidValue;
    if (b.src_rows && b.n_rows != b.nz) return cudaErrorInvalidValue;   // the reciprocal march stores every row
    const PipeShape sh = pipe_shape(b.nz);
    if (!sh.ca) return cudaErrorInvalidValue;
    void (*const kernel)(EikBatch, eikf::Dims, int, int*) =
        b.src_rows ? (sh.ca == 64 ? eik_pipe_recip_kernel<64, kPipeWarps> : eik_pipe_recip_kernel<128, kPipeWarpsDeep>)
                     : (sh.ca == 64 ? eik_pipe_kernel<64, kPipeWarps> : eik_pipe_kernel<128, kPipeWarpsDeep>);
    eikf::Dims D = fast_dims(b.nxmod, b.nz);
    // Lock-step columns in the box phase (a second column buffer per slice: 7 slices instead of 9 on the Example plane).
    // Kernel ms per launch at 1024 / 2048 / 4096 / 8192 chains with the box phase inlined: 7.70 / 13.99 / 26.42 / 51.07
    // against 8.03 / 14.24 / 26.66 / 51.07 with the per-lane in-place walk (profiles/README.md r2c).
    D.lock_cols = 1;
    const size_t slice = fast_smem_floats_per_warp(D) * sizeof(float);
    int dev = 0, sms = 148, smem_max = 232448;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    int n_slices = (int)(((size_t)smem_max - 256) / slice);
    if (n_slices > sh.warps) n_slices = sh.warps;
    if (n_slices < 2) return cudaErrorInvalidValue;
    const size_t smem = (size_t)n_slices * slice;
    // per instantiation and device: largest dynamic shared-memory size the kernel has been opted in for
    static size_t configured[4][64] = {};
    size_t* conf = (dev >= 0 && dev < 64) ? &configured[(sh.ca == 128) * 2 + (b.src_rows ? 1 : 0)][dev] : nullptr;
    if (!conf || smem > *conf) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (conf) *conf = smem;
    }
    const int n_tasks = (b.n_items * eik_sources(b) + 31) / 32;
    // per-warp global window: the scratch was sized for max_warps warps of the generic kernel
    const size_t have = (size_t)b.max_warps * eik_scratch_floats_per_warp(b.nxmod, b.nz);
    const long warps_by_scratch = (long)(have / fast_scratch_floats_per_warp(D));
    int blocks = (n_tasks + sh.warps - 1) / sh.warps;
    if (blocks > sms) blocks = sms;
    if ((long)blocks * sh.warps > warps_by_scratch) blocks = (int)(warps_by_scratch / sh.warps);
    if (blocks < 1) return cudaErrorInvalidValue;
    cudaError_t e = cudaMemsetAsync(task_counter, 0, sizeof(int), stream);
    if (e != cudaSuccess) return e;
    kernel<<<blocks, sh.warps * 32, smem, stream>>>(b, D, n_slices, task_counter);
    count_launch();
    return cudaGetLastError();
}

size_t eik_pipe_tie_floats(int nz)
{
    return (size_t)kPipeMaxCtas * (pipe_shape(nz).ca == 128 ? kPipeTieFloats<128> : kPipeTieFloats<64>);
}

int eik_fast_max_warps(int nxmod, int nz, int device)
{
    const eikf::Dims D = fast_dims(nxmod, nz);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    int per_sm = 0;
    const size_t smem = fast_smem_floats_per_warp(D) * sizeof(float);
    cudaFuncSetAttribute(eik_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaFuncSetAttribute(eik_fast_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, eik_fast_kernel, 32, smem);
    if (per_sm < 1) per_sm = 1;
    return sms * per_sm;
}

cudaError_t eik_launch_fast(const EikBatch& b, cudaStream_t stream)
{
    const int n_solves = b.src_iz ? b.n_solves : b.n_items * eik_sources(b);
    if (n_solves <= 0) return cudaSuccess;
    const eikf::Dims D = fast_dims(b.nxmod, b.nz);
    const size_t smem = fast_smem_floats_per_warp(D) * sizeof(float);
    static int configured_for = -1;
    int dev = 0;
    cudaGetDevice(&dev);
    static int resident = 0;
    if (configured_for != dev * 100000 + b.nz) {
        resident = eik_fast_max_warps(b.nxmod, b.nz, dev);
        configured_for = dev * 100000 + b.nz;
    }
    // scratch was sized for max_warps warps of the generic kernel, which is never less per warp
    const size_t have = (size_t)b.max_warps * eik_scratch_floats_per_warp(b.nxmod, b.nz);
    long warps = (long)(have / fast_scratch_floats_per_warp(D));
    if (warps > resident) warps = resident;
    // A launch with fewer warp-tasks than warps that can be resident lasts as long as one task, and a task is the shorter
    // the fewer lanes have to wait for each other in the box phase: spread it over the idle warps.
    int lpt = 32;
    while (lpt > 4 && ((long)n_solves + lpt / 2 - 1) / (lpt / 2) <= warps) lpt /= 2;
    const int n_tasks = (n_solves + lpt - 1) / lpt;
    if (warps > n_tasks) warps = n_tasks;
    if (warps < 1) warps = 1;
    eik_fast_kernel<<<(unsigned)warps, 32, smem, stream>>>(b, D, lpt);
    count_launch();
    return cudaGetLastError();
}

const char* eik_kernel_name(int which)
{
    static const char* names[kEikKernels] = {"eik_generic_kernel", "eik_fast_kernel", "eik_pipe_kernel", "eik_fine_kernel"};
    return (which >= 0 && which < kEikKernels) ? names[which] : "?";
}

size_t eik_fine_slice_floats_per_warp(int nxmod, int nz)
{
    return (size_t)eikf::gmem_floats_per_lane(fast_dims(nxmod, nz)) * 32;
}

cudaError_t eik_launch_fine(const EikBatch& b, cudaStream_t stream)
{
    const int n_solves = b.src_iz ? b.n_solves : b.n_items * eik_sources(b);
    if (n_solves <= 0) return cudaSuccess;
    if (!b.slice_scratch) return cudaErrorInvalidValue;
    const eikf::Dims D = fast_dims(b.nxmod, b.nz);
    const int n_tasks = (n_solves + 31) / 32;
    // one warp per CTA; the window (b.scratch) and the slice were sized for max_warps warps
    const size_t have = (size_t)b.max_warps * eik_scratch_floats_per_warp(b.nxmod, b.nz);
    long warps = (long)(have / fast_scratch_floats_per_warp(D));
    if (warps > b.max_warps) warps = b.max_warps;
    if (warps > n_tasks) warps = n_tasks;
    if (warps < 1) warps = 1;
    eik_fine_kernel<<<(unsigned)warps, 32, 0, stream>>>(b, D, 32);
    count_launch();
    return cudaGetLastError();
}

cudaError_t eik_launch(const EikBatch& b, cudaStream_t stream, int* which)
{
    int dummy;
    if (!which) which = &dummy;
    static int force_generic = -1;
    if (force_generic < 0) {
        const char* e = getenv("MCMCEQ_EIKONAL");
        force_generic = (e && strcmp(e, "generic") == 0) ? 1 : 0;
    }
    if (!force_generic && b.task_counter && b.tie_scratch && !b.src_iz && !b.full_out && (!b.src_rows || b.n_rows == b.nz) &&
        eik_pipe_supported(b.nxmod, b.nz)) {
        // worth it (and the per-warp scratch windows suffice) only when there is work for every warp of every SM
        const eikf::Dims D = fast_dims(b.nxmod, b.nz);
        const size_t have = (size_t)b.max_warps * eik_scratch_floats_per_warp(b.nxmod, b.nz);
        const long n_tasks = ((long)b.n_items * eik_sources(b) + 31) / 32;
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const int warps = pipe_shape(b.nz).warps;
        if ((long)(have / fast_scratch_floats_per_warp(D)) >= (long)sms * warps && n_tasks >= (long)sms * warps &&
            sms <= kPipeMaxCtas) {
            *which = kEikPipe;
            return eik_launch_pipe(b, b.task_counter, stream);
        }
    }
    if (!force_generic && eik_fast_supported(b.nxmod, b.nz)) { *which = kEikFast; return eik_launch_fast(b, stream); }
    if (!force_generic && b.slice_scratch && b.nxmod >= 2 && b.nz >= 2) { *which = kEikFine; return eik_launch_fine(b, stream); }
    *which = kEikGeneric;
    return eik_launch_generic(b, stream);
}

}  // namespace mq
