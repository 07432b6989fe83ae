// eikonal.cuh -- launch interface of the batched eikonal kernels (internal to the library).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace mq {

// One batch of independent solves on an nxmod x nz plane (reference: the nz calls of
// time_2d in setup_table_new, src/misfit.c:270-289, for many chains and both phases at once).
struct EikBatch {
    int nxmod, nz;
    // Work list.  Either "table mode": n_items slowness columns, every source depth of every
    // item is solved (n_solves = n_items*nz, solve g -> iz = g / n_items, item = g % n_items,
    // so that the lanes of a warp share the source depth and with it the sweep schedule), or
    // "list mode" (src_iz != nullptr): solve g uses column g and source depth src_iz[g].
    const float* slow;        // [n_items][nz] device, h / v per depth cell
    int n_items;
    const int32_t* n_items_dev; // table mode only: when non-null the item count is read on the device
                                // (n_items is then the upper bound the grid is sized for)
    const int32_t* src_iz;    // [n_solves] device or nullptr
    int n_solves;
    // Table mode only: optional execution order.  order[j] = the solve (iz * n_items + item) that lane j % 32 of warp
    // task j / 32 runs, or -1 (eik_order_tasks fills it: solves of one source depth that initialise and grow their
    // boxes alike are made neighbours so that the lanes of a warp stay in step).
    const int32_t* order;
    int32_t* task_counter;    // [1] device: work counter of the pipelined kernel (eik_launch_pipe), or nullptr
    float* tie_scratch;       // device, eik_pipe_tie_floats(nz) floats: per-CTA scratch of the pipelined kernel's tie fallback
    // Outputs (device).  full_out: [n_solves][nxmod*nz] in the reference layout (x*nz+y).
    float* full_out;
    // Receiver-row tables: table of item i starts at row_out[i] (or row_out_base + i*row_item_stride
    // when row_out == nullptr) and is laid out [n_rows][nz (source depth)][xpitch].
    float* const* row_out;
    float* row_out_base;
    size_t row_item_stride;
    const int32_t* rows;      // [n_rows] device: grid rows (receiver layers) that are kept
    int n_rows, xpitch;
    int32_t* status;          // [n_solves] device or nullptr
    int32_t* status_min;      // [1] device or nullptr: atomicMin of every solve's status
    // Scratch: per resident warp (nxmod*nz + kFineNodes) * 32 floats.
    float* scratch;
    int max_warps;
    // Planes that do not fit a shared-memory slice (eik_fine_kernel): eik_fine_slice_floats_per_warp() floats per warp for
    // max_warps warps, or nullptr (such planes then take the generic kernel).
    float* slice_scratch;
};

constexpr int kFineNodes = 22 * 43;   // refined grid of a left-edge source, src/time_2d.c:844-864

size_t eik_scratch_floats_per_warp(int nxmod, int nz);
// Generic one-lane-per-solve kernel, time field in global memory.
cudaError_t eik_launch_generic(const EikBatch& b, cudaStream_t stream);
// Warp-synchronous kernel, live state in shared memory (eik_fast.cuh).  Same EikBatch; its scratch need per warp
// is smaller (box window + refined grid) so the generic kernel's scratch always suffices.
bool eik_fast_supported(int nxmod, int nz);
cudaError_t eik_launch_fast(const EikBatch& b, cudaStream_t stream);
// The same warp-synchronous solver with its per-lane arrays in global memory, for planes of any size (the fine grid).
size_t eik_fine_slice_floats_per_warp(int nxmod, int nz);
cudaError_t eik_launch_fine(const EikBatch& b, cudaStream_t stream);
// One persistent CTA per SM: box phases on a pool of shared-memory slices, marches on a pool of TMEM sets; planes of up to
// 126 depth nodes.  eik_pipe_tie_floats(nz): size of EikBatch::tie_scratch for a plane of nz depth nodes.
bool eik_pipe_supported(int nxmod, int nz);
size_t eik_pipe_tie_floats(int nz);
cudaError_t eik_launch_pipe(const EikBatch& b, int* task_counter, cudaStream_t stream);
// Picks the kernel: pipelined when the launch fills the GPU and the plane fits a shared-memory slice, fused for smaller
// launches of such planes, generic otherwise (MCMCEQ_EIKONAL=generic forces the generic one).  *which (may be nullptr)
// receives the kernel taken, for mq_profile_kernels.
enum { kEikGeneric = 0, kEikFast = 1, kEikPipe = 2, kEikFine = 3, kEikKernels = 4 };
const char* eik_kernel_name(int which);
cudaError_t eik_launch(const EikBatch& b, cudaStream_t stream, int* which = nullptr);
// Regrouping of the solves of a table-mode batch (see EikBatch::order).  `work` holds the sort buffers:
// eik_order_bytes(max_solves) bytes.  Fills order[0 .. round_up(max_solves, 32)).
size_t eik_order_bytes(int max_solves);
cudaError_t eik_order_tasks(const EikBatch& b, int32_t* order, void* work, size_t work_bytes, cudaStream_t stream);
// resident warps the fast kernel can use on this device (for sizing the scratch)
int eik_fast_max_warps(int nxmod, int nz, int device);

}  // namespace mq
