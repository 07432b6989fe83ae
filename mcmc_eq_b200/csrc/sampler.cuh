// sampler.cuh -- device state of the Metropolis-Hastings sampler (chain.cu) that other translation units read: the
// sampler state save / load (state.cu) gathers and scatters it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "state.h"

namespace mq {

struct Snapshot {   // a full copy of a chain's state (the best model so far), SoA over chains
    int32_t* dim; float *z, *vp, *vpvs, *eq, *origin, *pres, *sres, *noise;
    double* rms; int64_t* number; int32_t* code; int32_t* flag;
};

// Decimated records (print_model_raw, src/mcmc_eq.c:234-248, written at :1163): a device-side ring of `slots` packed
// records per chain.  accept_kernel decides that the model just accepted is a record (pend), snapshot_kernel writes the
// chain's state into slot wr % slots and publishes it (wr + 1); a drain (pack_records_kernel, on the copy stream)
// copies the records [rd, wr) of every chain into a staging buffer and frees them (rd = wr).  A full ring drops the NEW
// record and counts it (lost): published slots are never overwritten, so a drain may run next to later steps.
// Record = kRecHead words of header (chain, code, dim, -, number as int64, rms as double), noise[8], z[md], vp[md],
// vpvs[md], eq[3 ne], origin[ne], pres[ns], sres[ns], padded to a multiple of four floats.
constexpr int kRecHead = 8;
struct Ring {
    float* data;          // [n][slots][rec_floats]
    int32_t *wr, *rd;     // [n] records published / handed to a drain so far
    int32_t* lost;        // [n] records dropped since the last drain
    int32_t* pend;        // [n] 0: nothing, 1: store the state as a record, 2: ring full (posterior accumulation only)
    int64_t* number; int32_t* code; double* rms;   // [n] header of the pending record
    int slots, rec_floats;
};
__host__ __device__ inline int rec_floats_of(int md, int ne, int ns) { return (kRecHead + 8 + 3 * md + 4 * ne + 2 * ns + 3) / 4 * 4; }

struct SamplerDev {
    int64_t *acce, *reject, *counts;
    uint64_t* draws;
    float* inv_control;
    int32_t *kind, *not_valid, *rebuilt;
    double* log_fac;
    float* noise_new;
    double* best_rms;
    float *wz, *wvp, *wvs;   // model_valid work arrays [n][md]
    Ring ring;
    Snapshot best;
    char *ps_start, *ps_main, *ps_over;
    int len_start, len_main, len_over;
    // replay mode (mq_replay_step): injected uniform deviates and per-chain results of the last decision
    float* u_inject;     // [n] or nullptr (every pass but a replayed one: the accept test draws from the chain's stream)
    float* r_alpha;      // [n]
    int32_t* r_accept;   // [n]
    double* r_newll;     // [n]
    int32_t* r_qidx;     // [n] injected event index of a Q proposal
    int32_t* r_dim;      // [n] injected number of nuclei of the proposed model
    // desynchronised stepping (mq_step): iterations a chain still owes to the current call, and what it does in the
    // current pass: 0 = evaluated and decided, 1 = idle, 2 = parked with a proposal that waits for its travel-time tables
    int32_t* todo;       // [n] or nullptr (lock-step passes)
    int32_t* hold;       // [n] or nullptr
    int32_t* pass_stat;  // [2] parked chains, chains that can still propose after this pass
};
}  // namespace mq
// One drain in flight (include/mcmceq_b200.h: mq_batch): device staging + pinned host copy of the packed records.
struct mq_batch {
    mq::Handle* h;
    int state;              // 0 free, 1 begun (pack kernel + count copy enqueued), 2 records on the host
    float* d_stage; int cap_records, rec_floats;
    int32_t *d_count, *h_count;     // [2] records, lost (device / pinned)
    float* h_stage; size_t h_cap_floats;   // pinned, grown on demand
    cudaEvent_t ev_count, ev_data;
    int n_records, n_lost;
    int delivered;          // records handed to the callback so far (a delivery that was stopped early can be resumed)
    std::vector<int>* order;
};
namespace mq {
struct Sampler : SamplerDev {
    std::string over_host;
    bool started;
    cudaStream_t copy_stream;
    cudaEvent_t ev_main;          // orders a drain behind the steps enqueued so far
    mq_batch batch[2];
    Snapshot cur;                 // scratch of mq_snapshot(which = 0)
    int32_t *todo_buf, *hold_buf, *stat_buf;   // storage of todo / hold / pass_stat, handed to the kernels by dev_desync() only
    float* u_buf;                              // storage of u_inject, handed to the kernels by dev_replay() only
    SamplerDev dev() const { return *this; }
    SamplerDev dev_desync() const { SamplerDev d = *this; d.todo = todo_buf; d.hold = hold_buf; d.pass_stat = stat_buf; return d; }
    SamplerDev dev_replay() const { SamplerDev d = *this; d.u_inject = u_buf; return d; }
};

// the handle's sampler, allocated on first use
int sampler_get(Handle* h, Sampler** out);

}  // namespace mq
