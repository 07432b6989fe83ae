// eikonal.cuh -- launch interface of the batched eikonal kernels (internal to the library).
//
// A caller describes the solves (EikBatch) and owns a work space (EikWork) that eik_work_alloc sized for its plane and
// batch size; eik_launch chooses the kernel and how many warps it runs with.  How much work space a kernel needs and
// which kernel a launch takes is decided in eikonal.cu alone.
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
    // Table mode only: reciprocal tables.  When non-null the sources of an item sit at the n_src_rows grid rows src_rows[rho]
    // instead of at every depth: n_solves = n_items*n_src_rows, solve g -> rho = g / n_items, item = g % n_items, and its
    // kept rows go to block rho of the item's table, row r at (rho*n_rows + r)*xpitch.  With rows = 0 .. nz-1 (the handle's
    // reciprocal mode) that is the [n_src_rows][nz][xpitch] layout of the parity table with its receiver-row and
    // source-depth axes swapped: t[x][y] of the source at row src_rows[rho] where parity has the time from (0, y) to
    // (x, src_rows[rho]) (by reciprocity T(a -> b) ~ T(b -> a)).  The pipelined kernel requires rows = 0 .. nz-1 then.
    const int32_t* src_rows;
    int n_src_rows;
    // Outputs (device).  Receiver-row tables: the table of item i starts at row_out[i] and is laid out
    // [n_rows][nz (source depth)][xpitch].  full_out: [n_solves][nxmod*nz] in the reference layout (x*nz+y).
    const int32_t* rows;      // [n_rows] device: grid rows (receiver layers) that are kept
    int n_rows, xpitch;
    float* const* row_out;
    // When row_out is null: the table of item i at row_out_base + i*row_item_stride.  No caller uses this form, but the
    // kernels keep its branch: without it nvcc 12.9 gives the fused and pipelined kernels 2 - 4 more registers and the
    // pipelined one about 140 more instructions (tools/sass_footprint.py), and the pipelined launch ran slower.
    float* row_out_base;
    size_t row_item_stride;
    float* full_out;
    int32_t* status;          // [n_solves] device or nullptr
    int32_t* status_min;      // [1] device or nullptr: atomicMin of every solve's status
    // Table mode only: run the solves in regrouped order when the work space has the sort buffers (solves of one source
    // depth that initialise and grow their boxes alike become neighbours, so that the lanes of a warp stay in step).
    bool regroup;
};

// Work space of the eikonal launches on one plane.  Callers allocate and free it and pass it to eik_launch; its fields
// are read by eikonal.cu only.
struct EikWork {
    int nxmod, nz;
    float* window;            // per-warp time-field windows: `warps` windows of the generic kernel's size (eikonal.cu)
    int warps;
    float* slices;            // planes that do not fit a shared-memory slice: per-warp arrays of eik_fine_kernel, or nullptr
    void* sort;               // regrouping (EikBatch::regroup): sort buffers and the execution order, or nullptr
    size_t sort_bytes;
    int32_t* order;
    int32_t* task_counter;    // pipelined kernel: work counter and per-CTA tie scratch, or nullptr
    float* tie;
    // launch facts of the plane on the device
    int sms;
    int fast_resident;        // warps of eik_fast_kernel that can be resident
    int pipe_ca, pipe_warps, pipe_slices;   // pipelined kernel: column-array length (0: not available), warps per CTA,
    size_t pipe_smem;                       // shared-memory slices per CTA and their bytes
};

// Allocates the work space of batches of up to max_solves solves on an nxmod x nz plane on `device` (the current device).
// tables: table rebuilds of a handle, which also get the regrouping sort and the pipelined kernel's buffers.  The window
// count is the warps of one full wave of max_solves, capped by a share of the free device memory (MCMCEQ_SCRATCH_FRACTION);
// the kernels loop over the solves with however many warps fit.  On failure nothing stays allocated.
cudaError_t eik_work_alloc(EikWork* w, int nxmod, int nz, int max_solves, bool tables, int device);
void eik_work_free(EikWork* w);

// Runs the batch on the work space of its plane: the pipelined kernel when the launch fills the GPU and the plane fits a
// shared-memory slice, the fused kernel for smaller launches of such planes, the fine-grid kernel for larger planes
// (MCMCEQ_EIKONAL=generic forces the generic one).  *which (may be nullptr) receives the kernel taken, for
// mq_profile_kernels.
enum { kEikGeneric = 0, kEikFast = 1, kEikPipe = 2, kEikFine = 3, kEikKernels = 4 };
const char* eik_kernel_name(int which);
cudaError_t eik_launch(const EikBatch& b, const EikWork& w, cudaStream_t stream, int* which = nullptr);

}  // namespace mq
