// state.h -- device-resident state of one handle (n_chains chains on one GPU).
//
// Data layout in HBM (all FP32 unless noted; n = n_chains, md = max_dim, ne = n_events,
// ns = n_stations, R = kept receiver rows, xp = xpitch >= nxmod):
//
//   model     z/vp/vpvs [2][n][md], dim [2][n]          double-buffered: mcur[c] = current buffer
//   eq        [n][ne][3]   pres/sres [n][ns]   noise [n][8]
//   tables    [2][n][2 phases][R][nz][xp]               double-buffered per chain AND phase: tcur[2c+ph]
//             only the receiver rows the misfit can ever read are kept (reference keeps all nz rows,
//             src/misfit.c:281-288; the values are the same, SURVEY.md section 7 H2-v); with reciprocal tables
//             (mq_set_tables) [R][nz][xp] is the field of a source at receiver row R read at every depth instead
//   evsum     [2][n][ne][8], origin [2][n][ne]          per-event class sums; ecur[c] = current buffer
//   mf [n][8], ll/rms/misfit [n] (double)               current likelihood
//
// Accept = flip an index, reject = nothing: the reference's table backup/restore copies
// (58 % of its CPU time, src/mcmc_eq.c:856,1161,1171) do not exist here.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mcmceq_b200.h"
#include "eikonal.cuh"

namespace mq {

// bits of the device error word Handle::err
constexpr int kErrStatcor = 1;   // a pick points to a station correction < -1000 (the reference exit()s, src/misfit.c:93,111)
constexpr int kErrRetry = 2;     // a start value could not be drawn inside its bounds (mq_init_chains)

struct DevPicks {
    int n_events, n_picks, max_event_picks;
    int32_t* ev_off;   // [ne+1]
    int32_t* n_p;      // [ne]
    int32_t* st_id;    // [np]
    int32_t* r0;       // [np] index of the pick's receiver layer in the kept rows (layer+1 is r0+1)
    int32_t* cp;       // [np] 2*class + (phase == S)
    float *x, *y, *t, *w1, *w2;   // [np]
    // the same per pick in two vector loads (misfit_kernel): rec4 = (x, y, t, w1), rec2 = (w2, bits of st_id | r0 << 20 | cp << 28)
    float4* rec4;      // [np]
    float2* rec2;      // [np]
    double* fix;       // [ne*3]
};

// What a misfit evaluation reads and where it writes: either the current state
// (mq_forward) or a proposal (mq_step).  All arrays are per chain.
struct EvalView {
    int32_t* mbuf;     // [n]   model buffer to evaluate
    int32_t* tbuf;     // [2n]  table buffer per phase to evaluate with
    int32_t* ebuf;     // [n]   evsum/origin buffer to write
    int32_t* q_idx;    // [n]   event whose hypocentre is overridden by q_xyz (-1: none)
    float* q_xyz;      // [n][3]
    int32_t* r_idx;    // [n]   station whose correction is perturbed (-1: none; -2: take pres_over/sres_over instead)
    float* r_d;        // [n][2] dP, dS of the perturbation
    int32_t* ev_only;  // [n]   >= 0: evaluate only this event (result in evq/oq); -1: all; -2: none
    float* pres_over;  // [n][ns] proposed station corrections given in full (replay mode, mq_replay_step) or nullptr
    float* sres_over;
    const int32_t* hold;   // [n] or nullptr: chains with hold[c] != 0 are not evaluated in this pass (desynchronised stepping, chain.cu)
};

// On-device posterior accumulation = pass 1 of the reference's analyse_eq (src/analyse_eq.c:496-643) applied to every
// decimated model as it is produced.  Two contiguous blocks so that the cross-GPU reduction is one all-reduce each.
struct Posterior {
    int on;
    float dv, dvpvs;
    int ndv, ndvpvs;
    long long burn_in;      // models with number <= burn_in are skipped (the scripts' `$3 > bi` filter)
    int32_t* iblock;        // hist_vp [ndv][nz] | hist_vpvs [ndvpvs][nz] | boundary [nz]
    double* dblock;         // vsum [nz][4] | eqsum [ne][8] | ressum [ns][4] | noisesum [16] | n_models [1]
    size_t n_int, n_dbl;
};

// On-device convergence diagnostics (diag.cu, DESIGN.md section 4d): per chain and posterior quantity, batch sums of
// d = x - ref over the same decimated models the posterior takes, in K slots whose length doubles when they are full.
// Memory: (2K + 1) Q doubles + 16 bytes per chain, Q = 10 + 2 nz + 4 ne + 2 ns quantities.
struct Diag {
    int on;
    int K, Q;               // batch slots (n_batches), quantities
    long long burn_in;      // models with number <= burn_in are skipped, as in the posterior
    double* ref;            // [n][Q] the chain's first used model
    double* sum;            // [n][K][Q] sums of d per batch slot
    double* sumsq;          // [n][K][Q] sums of d*d
    int64_t* n_models;      // [n] used models so far
    int32_t* batch_len;     // [n] models per full batch (L)
    int32_t* full_batches;  // [n] full batches (k); slot k is the open one
    double* scratch;        // summary work space (diag.cu), allocated on the first mq_diag_summary
    size_t scratch_bytes;
};

// On-device hypocentre uncertainty (hypo.cu, DESIGN.md section 4e): per chain and event, sums of d = v - ref and of the
// ten products d_i d_j of v = (x, y, z, t) over the same decimated models the posterior takes, and per event histograms
// of x, y and z over the hypocentre box.  Memory: 18 doubles per (chain, event).
struct Hypo {
    int on;
    float bin;              // bin width (km)
    int nb[3];              // bins of x, y, z
    long long burn_in;      // models with number <= burn_in are skipped, as in the posterior
    int32_t* hist;          // [ne][nb[0] + nb[1] + nb[2]]
    int32_t* outside;       // [ne][3] values outside the box (clamped into the end bins)
    double* ref;            // [n][4][ne] the chain's first used value
    double* sum;            // [n][4][ne] sums of d
    double* cross;          // [n][10][ne] sums of d_i d_j (xx xy xz xt yy yz yt zz zt tt)
    int64_t* n_models;      // [n] used models so far
    void* scratch;          // summary work space (hypo.cu), allocated on the first mq_hypo_summary
    size_t scratch_bytes;
};

struct Handle {
    mq_config cfg;
    int device;
    cudaStream_t stream;
    int n, md, ne, ns, np;
    int nz, nxmod, xp, n_rows;
    float inv_control;   // sign as currently active (negative = no low-velocity zones)
    int lvz_flag;
    int n_class[8];
    int sum_of_picks;
    float xmin, xmax, ymin, ymax, zmin, zmax;
    size_t tab_stride;   // floats per (chain, phase) table
    uint64_t seed;
    uint64_t picks_sum;  // checksum of the picks as mq_create received them (state.cu: a saved state belongs to them)
    bool models_set, forward_done;
    int tables_mode;     // MQ_TABLES_PARITY or MQ_TABLES_RECIPROCAL (mq_set_tables): how table rebuilds solve (eikonal.cuh)

    DevPicks pk;
    int32_t* d_rows;     // [n_rows] kept grid rows
    int32_t* rows_host;  // [n_rows] (malloc)
    int32_t* d_all_rows; // [nz] 0 .. nz-1: the rows a reciprocal table rebuild keeps

    // chain state
    int32_t *dim, *mcur, *tcur, *ecur;
    float *z, *vp, *vpvs;
    float *eq, *pres, *sres, *noise;
    float* tab;
    float *evsum, *origin;
    float* mf;           // [n][8]
    double *ll, *rms, *misfit;
    int32_t* err;        // [1] device error word (bits kErrStatcor, kErrRetry)
    int32_t* host_flags; // pinned [2]: copies of err and solve_status made at the end of an asynchronous call ...
    cudaEvent_t flags_ev; // ... valid once this event has completed
    bool flags_pending;
    cudaEvent_t timer_ev[2][16];   // mq_timer

    // evaluation plumbing
    EvalView cur_view;   // view of the current state
    EvalView prop_view;  // view of the proposal (mq_step)
    float *evq, *oq;     // [n][8], [n] single-event results
    float* mf_eval;      // [n][8] totals of the last evaluation
    float* resid;        // [n][np] per-pick scratch, or nullptr: allocated when predictions are wanted or an event has more than 256 picks
    float* tpred;        // [n][np] or nullptr (allocated on first mq_get_predictions)
    bool want_pred;

    // eikonal work lists
    int32_t* item_chain; // [2n] chain of each rebuild item
    int32_t* item_phase; // [2n]
    int32_t* n_items;    // [1] device counter
    float* slow;         // [2n][nz]
    float** item_tab;    // [2n] destination table of each item
    int32_t* solve_status; // [1] min over solves
    EikWork eik;         // work space of the table rebuilds (eikonal.cuh), for 2n*nz solves

    // sampler (chain.cu)
    void* sampler;
    int ring_slots;      // records per chain of the device-side output ring (mq_set_ring; 0 = default)

    // optional timing of the dominant kernel (mq_profile): CUDA events round every eikonal launch
    void* prof;

    // multi-GPU (comm.cu): global index of chain 0, inverse temperatures, NCCL communicator, posterior accumulators
    long long chain_offset;
    float* beta;         // [n] or nullptr (all 1)
    void* comm;
    Posterior post;
    Diag diag;
    Hypo hypo;
};

// checksums a saved sampler state carries (state.cu)
uint64_t config_checksum(const mq_config* cfg);
uint64_t picks_checksum(const mq_picks* pk);

// diagnostics (diag.cu): number of quantities of a handle; allocate (zeroed) / free the accumulators
inline int diag_quantities(int nz, int ne, int ns) { return 10 + 2 * nz + 4 * ne + 2 * ns; }
int diag_alloc(Handle* h, int K, long long burn_in);
void diag_destroy(Handle* h);
// hypocentre accumulators (hypo.cu): bins per axis for a bin width (-1: more than 2^20 on some axis); allocate (zeroed) /
// free them
int hypo_bins(const Handle* h, float bin_km, int nb[3]);
int hypo_alloc(Handle* h, float bin_km, long long burn_in);
void hypo_destroy(Handle* h);
// comm.cu: in-place sum of `count` doubles (int32s) over the ranks of the handle's communicator; nothing without one
int comm_allreduce_sum(Handle* h, double* buf, size_t count);
int comm_allreduce_sum(Handle* h, int32_t* buf, size_t count);

}  // namespace mq

struct mq_handle {
    mq::Handle h;
};
