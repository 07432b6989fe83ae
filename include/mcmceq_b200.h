/* mcmceq_b200.h -- C ABI of libmcmceq_b200.so, the B200 implementation of mcmc_eq's
 * forward-model / likelihood hot path.
 *
 * Plain C: pointers and sizes only, every entry point returns an int status
 * (0 = MQ_OK, negative = error) and never calls exit().  The reference has no FFI;
 * its seams for this path are four C functions plus the process command line
 * (SURVEY.md section 8b).  Each entry point below names the reference interface it
 * replaces.  All pointer arguments are HOST pointers unless the name ends in _dev.
 *
 * Thread-safety: a handle may be used by one host thread at a time; different handles
 * (e.g. one per GPU) are independent.  The reference's time_2d keeps file-scope
 * statics (src/time_2d.c:219-259) and is not re-entrant; this library is.
 */
#ifndef MCMCEQ_B200_H
#define MCMCEQ_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MQ_OK 0
#define MQ_ERR_ARG (-1)          /* bad argument / size                                          */
#define MQ_ERR_CUDA (-2)         /* CUDA runtime error, see mq_last_error()                       */
#define MQ_ERR_UNSUPPORTED (-3)  /* call pattern outside the hot path (see mq_time_2d)            */
#define MQ_ERR_SOLVER (-4)       /* at least one eikonal solve reported a negative status         */
#define MQ_ERR_STATCOR (-5)      /* a pick points to an invalid station correction (< -1000);
                                    the reference prints and exit(0)s, src/misfit.c:93,111         */
#define MQ_ERR_NOMEM (-6)
#define MQ_ERR_STATE (-7)        /* call made in the wrong order                                  */
#define MQ_ERR_RETRY (-8)        /* a start value could not be drawn inside its bounds (the reference's
                                    rand_gauss_bounded would loop for ever, src/mcmc_eq.c:149-159)  */
#define MQ_ERR_BUSY (-9)         /* both drain batches are in flight (mq_drain_begin)             */

#define MQ_MAX_CLASSES 8         /* 4 pick classes x {P,S}: index = 2*class + (phase == S)        */

/* ---- grid: reference struct GRDHEAD, src/mc.h:91-100 ------------------------------ */
typedef struct mq_grid {
    float h;            /* mesh spacing (km)                                    */
    int32_t nx, ny, nz; /* nodes; the eikonal plane is nxmod x nz,              */
                        /* nxmod = (int)sqrt(nx*nx+ny*ny)  (src/mcmc_eq.c:520)  */
    float x0, y0, z0;
} mq_grid;

/* ---- sampler settings: the 41 lines of config_eqx.dat, src/mcmc_eq.c:345-388 ------ */
typedef struct mq_config {
    mq_grid grid;
    int32_t max_dim;                       /* line 8  */
    float vpmin, vpmax, vpvsmin, vpvsmax;  /* 9-12    */
    float noise_min, noise_max;            /* 13-14   */
    float residual_min, residual_max;      /* 15-16   */
    float sdevx, sdevy, sdevz;             /* 17-19 (17,18 unused by the reference; 19 = nucleus move) */
    float sdevvp, sdevvpvs, sdevn;         /* 20-22   */
    float sdevxs, epi_search;              /* 23      */
    float sdevys, sdevzs, sdevresidual;    /* 24-26   */
    float inv_control;                     /* 27, as written in the file (sign = LVZ switch) */
    int32_t reference_station, scor_flag;  /* 28      */
    float ref_statcor_P, ref_statcor_S;    /* 28      */
    int32_t tria;                          /* 29: 0 = Voronoi cells, 1 = linear gradients between nuclei */
    int32_t j_max_start, j_max_main;       /* 30      */
    int32_t deci;                          /* 31      */
    int32_t true_random, eikonal;          /* 32      */
    char dstring_start[64], dstring_main[64]; /* 33   */
    int32_t aflag;                         /* 34 */
    char inp_model_switch[16];             /* 34 */
    float start_vp, sdev_start_vp, start_vp_grad; /* 36 */
    float start_vpvs, sdev_start_vpvs;     /* 37 */
    int32_t start_cell_number, sdev_start_cell_number; /* 38 */
    float start_noise;                     /* 39 */
    float start_delay, sdev_start_delay;   /* 40 */
    float r_start_eqh, r_start_eqv;        /* 41 */
} mq_config;

/* ---- picks: reference struct OBS / struct DATA (src/mc.h:102-134), flattened ------
 * Picks of event e are [ev_off[e], ev_off[e+1]); inside an event all P picks come first,
 * then all S picks, each in file order -- the order the reference sums them in
 * (src/misfit.c:87-119). */
typedef struct mq_picks {
    int32_t n_events, n_picks, n_stations;
    const int32_t* ev_off;   /* [n_events+1]                                        */
    const int32_t* n_p;      /* [n_events] number of P picks of the event           */
    const int32_t* st_id;    /* [n_picks]                                           */
    const float* x;          /* [n_picks] station coordinates (km)                  */
    const float* y;
    const float* z;
    const float* t;          /* [n_picks] observed travel time rel. to reftime (s)  */
    const int32_t* cls;      /* [n_picks] pick class 0..3                           */
    const double* reftime;   /* [n_events]                                          */
    const double* fix;       /* [n_events*3] fixed x,y,z or -9999 (src/mcmc_eq.c:610-612) */
} mq_picks;

/* ---- chain state: SoA mirror of reference struct Model, src/mc.h:68-89 ------------ */
typedef struct mq_models {
    int32_t n_chains, max_dim, n_events, n_stations;
    int32_t* dim;      /* [n_chains]                      Model.dimension */
    float* z;          /* [n_chains*max_dim]              Model.z         */
    float* vp;         /* [n_chains*max_dim]              Model.vp        */
    float* vpvs;       /* [n_chains*max_dim]              Model.vpvs      */
    float* eq;         /* [n_chains*n_events*3] x,y,z     Model.eq        */
    float* pres;       /* [n_chains*n_stations]           Model.pres      */
    float* sres;       /* [n_chains*n_stations]           Model.sres      */
    float* noise;      /* [n_chains*8] index 2*class+phase (p_noise0,s_noise0,p_noise1,...) */
    float* origin;     /* [n_chains*n_events] (output)    Model.origin    */
} mq_models;

typedef struct mq_handle mq_handle;

const char* mq_version(void);
/* Text of the last error raised on the calling thread. */
const char* mq_last_error(void);
/* Number of CUDA kernels this library has launched since it was loaded (bench.py's gpu_launches). */
int64_t mq_launch_count(void);

/* ===== unit-testable twins of the reference functions ================================ */

/* Drop-in for   int time_2d(float*hs,float*t,int nx,int ny,float xs,float ys,float eps,int msg)
 * (reference src/fdtimes.h:6-7, src/time_2d.c:301).  Same argument meaning and array layout
 * (x-major, index x*ny+y), one solve on the GPU.  Only the call pattern of the hot path is
 * implemented: hs constant along x (src/misfit.c:257-266), xs == 0, ys an integer node,
 * eps_init == 0.001f; anything else returns MQ_ERR_UNSUPPORTED and leaves t untouched.
 * Unlike the reference, hs is never written to. */
int mq_time_2d(const float* hs, float* t, int nx, int ny, float xs, float ys, float eps_init, int messages);

/* Batched form: n independent solves on an nxmod x nz plane.  slow[i*nz + k] is h/v of depth
 * cell k (what src/misfit.c:263 writes into every column of hsbuf), src_iz[i] the source depth
 * node.  t_out[i] receives the full field in the reference layout (nxmod*nz floats, index
 * x*nz+y); status[i] (may be NULL) the per-solve code (0 or negative). */
int mq_eikonal_batch(const float* slow, const int32_t* src_iz, int n, int nxmod, int nz, float* t_out,
                     int32_t* status, int device);

/* Drop-in for   float traveltimet(float **ttt, int nx, int ny, int nz, float h, float dist, float z, float z0)
 * (reference src/interpol.c:43-83): bilinear interpolation of one receiver layer of a HOST table, ttt[iz][ix] with
 * iz the source-depth node and ix the distance node (nx, ny are the grid's horizontal node counts, the table has
 * (int)sqrt(nx^2 + ny^2) distance nodes, :52); 1e30 outside the table (:64-65).  The four corner values travel to
 * the device and the library's own lookup code (the one misfit_kernel uses for every pick) evaluates them, so this
 * entry point is the unit-testable twin of that code, not a second implementation.  *t_out receives the time. */
int mq_traveltimet(float* const* ttt, int nx, int ny, int nz, float h, float dist, float z, float z0, float* t_out, int device);

/* ===== batched sampler ==================================================================
 * One handle drives n_chains chains on one GPU.  Model state, travel-time tables and RNG
 * state stay on the device between calls. */
int mq_create(const mq_config* cfg, const mq_picks* picks, int n_chains, int device, uint64_t seed,
              mq_handle** out);
int mq_destroy(mq_handle* h);

/* Upload / download chain states (host SoA <-> device). */
int mq_set_models(mq_handle* h, const mq_models* m);
int mq_get_models(mq_handle* h, mq_models* m);

/* Batched drop-in for cal_fit_newx (reference src/misfit.c:45-161) on the models currently in
 * the handle: calct = 0 none, 1 P tables, 2 S tables, 3 both are rebuilt first
 * (setup_table_new, src/misfit.c:165-293), then the residual sums of squares per pick class
 * (mf[chain*8 + 2*class + phase], the reference's *mfp0,*mfs0,*mfp1,...) and the origin times
 * (origin[chain*n_events + e] = Model.origin) are computed.  mf / origin may be NULL. */
int mq_forward(mq_handle* h, int calct, float* mf, float* origin);

/* Same, for models passed in host memory: upload, forward, download -- the end-to-end call. */
int mq_forward_host(mq_handle* h, const mq_models* m, int calct, float* mf, float* origin);

/* For a host-driven loop built on mq_forward_host (the reference's own main): after mq_forward_host the device tables
 * are those of the last call with calct != 0, exactly like the reference's tttpr/tttsr.  mq_tables_save /
 * mq_tables_restore are the reference's backup and restore of them (the triple loops at src/mcmc_eq.c:856,1161 and
 * :1171), as device-to-device copies.  Not needed with mq_step, which flips buffers instead. */
int mq_tables_save(mq_handle* h);
int mq_tables_restore(mq_handle* h);
/* The same for the tables of one phase only: phases = 1 (P), 2 (S) or 3 (both).  A 'V' proposal rebuilds the S table
 * alone (calct = 2, src/mcmc_eq.c:975) while the P table stays. */
int mq_tables_save_phases(mq_handle* h, int phases);
int mq_tables_restore_phases(mq_handle* h, int phases);

/* Full travel-time table of one chain in the reference layout ttt[nz][nz][nxmod]
 * (ttt[j][iz][i], src/misfit.c:281-288); phase 1 = P, 2 = S.  Recomputes that chain's table
 * with every receiver row kept; meant for parity tests and the setup_table_new shim. */
int mq_get_table(mq_handle* h, int chain, int phase, float* ttt);
/* The receiver rows of that table as they are stored on the device (what cal_fit_newx can ever read of it,
 * src/misfit.c:91,109): rows_out[r][iz][i] = ttt[row_index[r]][iz][i], r < n_rows.  Returns n_rows (>= 0) or a negative
 * status; either output may be NULL (call with both NULL to learn n_rows). */
int mq_get_rows(mq_handle* h, int chain, int phase, float* rows_out, int32_t* row_index);

/* How the travel-time tables are built (opt-in fast mode).  MQ_TABLES_PARITY (the default): one solve per source depth,
 * nz per (chain, phase) table, as the reference does (src/misfit.c:270-289).  MQ_TABLES_RECIPROCAL: one solve per stored
 * receiver row, with the source at that row, and the event depth read off its field: rows_out[r][iz][i] of mq_get_rows
 * is then the time from a source at (0, row_index[r]) to node (i, iz), used as the time from (0, iz) to (i, row_index[r]).
 * n_rows solves instead of nz (3 instead of 62 on the Example grid).  The finite-difference scheme is not exactly
 * reciprocal, so predictions differ from the parity mode's: DESIGN.md section 6 gives the measured error.  mq_forward,
 * mq_forward_host, mq_step, mq_replay_step and the rebuild in mq_state_load follow the mode; mq_get_table gives
 * MQ_ERR_UNSUPPORTED (no parity table exists).  No effect with eikonal == 0 or aflag == 1.  Call before mq_set_models /
 * mq_init_chains / mq_state_load: MQ_ERR_STATE afterwards; MQ_ERR_ARG for any other mode. */
#define MQ_TABLES_PARITY 0
#define MQ_TABLES_RECIPROCAL 1
int mq_set_tables(mq_handle* h, int mode);

/* Per-pick predictions of one chain after mq_forward: what cal_fit_newx prints with out=1
 * (src/misfit.c:130-143).  resid / tpred are [n_picks] in the handle's pick order. */
int mq_get_predictions(mq_handle* h, int chain, float* resid, float* tpred);

/* Sampler: random start models (src/mcmc_eq.c:559-630) + first forward (:739-765). */
int mq_init_chains(mq_handle* h);
/* n_iters Metropolis-Hastings iterations of every chain (src/mcmc_eq.c:845-1192) with the
 * device RNG.  proposal_override: NULL = the config's balanced proposal strings
 * (src/mcmc_eq.c:769-834), else a string of proposal letters to draw from uniformly. */
int mq_step(mq_handle* h, int n_iters, const char* proposal_override);

/* ---- replay: one iteration driven by a recorded proposal stream instead of the device RNG -------------------
 * The second correctness level of the path: the reference's own proposals (recorded from the unmodified reference,
 * oracle/replay_log.c) are scored by this library and its accept/reject decisions compared with the reference's.
 * For chain c: kind[c] is the arm of the proposal switch (src/mcmc_eq.c:866-1130; 0 = leave the chain alone),
 * `proposed` holds the complete proposed state -- the arm decides what is read: dim/z/vp/vpvs for P V M B D, event
 * q_idx[c] of eq for Q, pres/sres for R, noise for N --, log_fac[c] the proposal-ratio term (:1038,1070,1114),
 * u[c] the uniform deviate of the accept test (:1141).  What mq_step does after drawing a proposal happens
 * unchanged: table rebuild by calct, misfit, alpha12 = min(1, nexp(log_fac + new_ll - old_ll)), accept iff
 * u < alpha12, buffer flips, counters, decimated records.  Outputs (any may be NULL): accepted[c], alpha[c],
 * new_ll[c], mf[c*8 + 2*class+phase] = class sums of the proposal. */
typedef struct mq_replay {
    int32_t n_chains;
    const char* kind;            /* [n_chains] */
    const mq_models* proposed;
    const int32_t* q_idx;        /* [n_chains] (read for 'Q' only; may be NULL when no chain proposes Q) */
    const double* log_fac;       /* [n_chains] */
    const float* u;              /* [n_chains] */
    int32_t* accepted;
    float* alpha;
    double* new_ll;
    float* mf;
} mq_replay;
int mq_replay_step(mq_handle* h, const mq_replay* r);

/* Per-chain statistics (device -> host). counts[chain*20 + i]: 0 tested(nmod), then a/r pairs
 * for N,P,V,Q,R,M,B,D in the order of the reference's cnt lines (src/mcmc_eq.c:1199-1207),
 * 17 accepted, 18 rejected. */
int mq_get_stats(mq_handle* h, int64_t* counts, double* loglik, double* rms);

/* ---- records: what print_model_raw writes (src/mcmc_eq.c:234-248) ------------------------- */
#define MQ_REC_MODEL 0    /* decimated accepted model  ("mod", every deci-th accepted, :1163) */
#define MQ_REC_BEST 1     /* best-RMS model so far     ("bat BF", :1186-1196)                 */
#define MQ_REC_CURRENT 2  /* current state of the chain ("sta ST" right after mq_init_chains, :763) */
typedef struct mq_record {
    int32_t chain, kind;
    char code;            /* proposal letter that produced the model: Q R P V M B D N ('S' start, 'F' best) */
    int64_t number;       /* Model.number */
    int32_t dim;
    double rms;
    const float *noise;   /* [8] index 2*class+phase */
    const float *z, *vp, *vpvs;        /* [dim]           */
    const float *eq, *origin;          /* [n_events*3], [n_events] */
    const float *pres, *sres;          /* [n_stations]    */
} mq_record;
/* Called once per record; pointers are valid during the call only.  Return non-zero to stop: records not yet delivered stay
 * in their batch (a further mq_batch_deliver call continues with them; the synchronous mq_drain discards them). */
typedef int (*mq_record_fn)(void* user, const mq_record* rec);

/* Decimated records wait in a device-side ring of `slots` records per chain (default 4, 1..64; MCMCEQ_RING_SLOTS
 * overrides the default).  A chain whose ring is full drops the new record and counts it as lost; a ring of R slots
 * therefore survives R * deci iterations between two drains.  Call before mq_init_chains / the first mq_step. */
int mq_set_ring(mq_handle* h, int slots);

/* Synchronous drain: hands every pending decimated record to fn (the records of a chain in the order they were
 * produced) and frees their ring slots.  *n_lost (may be NULL) = records dropped since the previous drain. */
int mq_drain(mq_handle* h, mq_record_fn fn, void* user, int* n_lost);

/* Asynchronous drain, the output path for thousands of chains (the reference writes 1 + noq + nos lines per record,
 * src/mcmc_eq.c:234-248, from the sampling loop itself, :1163).  mq_drain_begin enqueues -- on a second stream, behind
 * the steps issued so far -- a kernel that packs the pending records into a staging buffer and frees their ring slots;
 * it returns at once and later mq_step calls run next to it.  The batch then belongs to the caller and may be used from
 * ANY host thread (a writer thread), while the handle goes on stepping: mq_batch_wait blocks until the records are in
 * pinned host memory (one cudaMemcpyAsync of exactly the packed records), mq_batch_deliver calls fn once per record,
 * mq_batch_release gives the batch back.  A handle owns two batches; MQ_ERR_BUSY when both are in flight. */
typedef struct mq_batch mq_batch;
int mq_drain_begin(mq_handle* h, mq_batch** batch);
int mq_batch_wait(mq_batch* batch, int* n_records, int* n_lost);
int mq_batch_deliver(mq_batch* batch, mq_record_fn fn, void* user);
int mq_batch_release(mq_batch* batch);

/* which = 0: current state of `chain`, 1: its best-RMS model so far.  mq_snapshot_all: the same for every chain of the
 * handle with bulk copies (fn is called n_chains times, chain 0 first). */
int mq_snapshot(mq_handle* h, int chain, int which, mq_record_fn fn, void* user);
int mq_snapshot_all(mq_handle* h, int which, mq_record_fn fn, void* user);

int mq_sync(mq_handle* h);

/* ===== more than one GPU =====================================================================================
 * One process per GPU, chains sharded contiguously (the reference runs chains as independent processes,
 * run/srun_mcmc_eq.sh:13,35): the data path has no collective.  NCCL appears in two optional places. */

/* Global index of this handle's chain 0.  Chain g of a job draws from the random stream (seed, g) whichever GPU it
 * runs on, so a run is reproducible under any sharding.  Call before mq_init_chains.  mq_comm_init sets rank*n_chains. */
int mq_set_chain_offset(mq_handle* h, int64_t first_chain);

/* On-device posterior accumulation = pass 1 of the reference's analyse_eq (src/analyse_eq.c:496-643) applied to every
 * decimated model (the "mod" records, src/mcmc_eq.c:1163) whose number is > burn_in, as it is produced:
 *   hist_vp[j*nz + i]   models whose Vp at depth node i falls in bin j, j = (int)((v - vpmin)/dv)   (hcountp, :589-590)
 *   hist_vpvs[j*nz + i] the same for Vp/Vs (hcounts, :605-606);  boundary[i] models with a layer boundary at node i (:586)
 *   vsum[i*4 + k]       sums over models of vp, vp^2, vpvs, vpvs^2 at node i (values clipped to the prior range, :587-588)
 *   eqsum[e*8 + k]      sums of x, y, z, origin time of event e, then of their squares (:619-623)
 *   ressum[s*4 + k]     sums of the P and S correction of station s, then of their squares (:636-637)
 *   noisesum[k], noisesum[8 + k]   sums of the eight sigmas (index 2*class+phase) and of their squares (:525-532)
 * mq_posterior_begin allocates and zeroes the accumulators (dims tells the sizes), mq_posterior_get copies them out
 * (any pointer may be NULL), mq_posterior_allreduce sums them over all ranks of the communicator in place. */
typedef struct mq_posterior_dims { int32_t ndv, ndvpvs, nz, n_events, n_stations; } mq_posterior_dims;
int mq_posterior_begin(mq_handle* h, float dv, float dvpvs, int64_t burn_in, mq_posterior_dims* dims);
int mq_posterior_get(mq_handle* h, int32_t* hist_vp, int32_t* hist_vpvs, int32_t* boundary, double* vsum, double* eqsum,
                     double* ressum, double* noisesum, int64_t* n_models);
int mq_posterior_allreduce(mq_handle* h);

/* Convergence diagnostics on the device: split R-hat and a batch-means effective sample size (ESS) of every quantity the
 * posterior summarises, from the same used models (decimated, number > burn_in; a model dropped from a full ring counts).
 * Q = 10 + 2 nz + 4 n_events + 2 n_stations quantities, in this order: 0 rms, 1 dim, 2..9 the sigmas (2*class+phase),
 * Vp at each depth node, Vp/Vs at each depth node (the values mq_posterior_* bins: nearest nucleus or, with TRIA = 1, the
 * interpolated profile, clipped to the prior range), x y z t of each event ([event][4]), P and S correction of each
 * station ([station][2]).  Every chain with any temperature beta counts, as in the posterior.
 *
 * Per chain: ref[q] = the chain's first used model; K = n_batches slots (even, 8 .. 64) of sums of d = (double)x - ref and
 * of d*d (round to nearest, no contraction); a slot holds batch_len models (L, starting at 1).  When the open slot is full
 * full_batches (k) grows; when k reaches K, slot i = slot 2i + slot 2i+1 (i ascending), slots K/2 .. K-1 are zeroed,
 * k = K/2 and L doubles.  Memory: (2K + 1) Q doubles + 16 bytes per chain (K = 16, config 3: 280 MB; config 4: 18 GB),
 * plus 2 Q doubles per chain of work space on the first mq_diag_summary.
 *
 * Summary, over the chains with k >= 4 (chains_used): split R-hat from sequences A = batches [0, h) and B = [h, 2h),
 * h = k/2; n_j = h L, m_j = S_j/n_j, s_j^2 = (T_j - S_j m_j)/(n_j - 1), mu_j = ref + m_j; over the M = 2 chains_used
 * sequences W = mean s_j^2, Bv = sum (mu_j - mean mu)^2 / (M - 1), var+ = (nbar - 1)/nbar W + Bv, rhat = sqrt(var+/W).
 * ESS: y_cb = S_cb / L_c over all k_c full batches, sigma2 = sum_c L_c sum_b (y_cb - ybar_c)^2 / sum_c (k_c - 1),
 * N = sum_c k_c L_c, ess = N var+ / sigma2.  mean = sum_c (k_c L_c ref_c + sum_b S_cb) / N, sd = sqrt(var+).  No used
 * chain: everything NaN; var+ == 0: rhat and ess NaN; W == 0 < var+: rhat +inf; sigma2 == 0 < var+: ess +inf.
 *
 * mq_diag_begin allocates and zeroes the accumulators (again = restart), before or after mq_init_chains; MQ_ERR_ARG for a
 * negative burn_in or a bad n_batches.  mq_diag_chains copies the raw accumulators out (any pointer may be NULL): ref
 * [n_chains][Q], sum and sumsq [n_chains][K][Q], batch_len, full_batches, n_models [n_chains].  mq_diag_summary computes the
 * summary on the device (fixed-order reductions, no floating-point atomics: the same accumulators give the same bits);
 * mean .. ess are [Q], *n_models = N and *chains_used one each (any may be NULL).  With collective != 0 and a communicator
 * (mq_comm_init) the sums are all-reduced over the ranks in two rounds and every rank gets the job-wide numbers; without
 * one, collective is ignored.  It first reports a pending error of an earlier asynchronous call.  Both return MQ_ERR_STATE
 * before mq_diag_begin.  The accumulators are part of a saved state (MQ_STATE_DIAG). */
typedef struct mq_diag_dims { int32_t n_quantities, nz, n_events, n_stations, n_batches; } mq_diag_dims;
int mq_diag_begin(mq_handle* h, int64_t burn_in, int n_batches, mq_diag_dims* dims);
int mq_diag_chains(mq_handle* h, double* ref, double* sum, double* sumsq, int32_t* batch_len, int32_t* full_batches,
                   int64_t* n_models);
int mq_diag_summary(mq_handle* h, int collective, double* mean, double* sd, double* rhat, double* ess, int64_t* n_models,
                    int32_t* chains_used);

/* Hypocentre uncertainty on the device: per event the mean, the 4 x 4 covariance of (x, y, z, t), quantiles and mode of
 * x, y and z, and the error ellipsoid of (x, y, z), from the same used models as mq_posterior_* and mq_diag_* (decimated,
 * number > burn_in; a model dropped from a full ring counts; every chain whatever its beta).  t is the model's origin time.
 * These are this library's own statistics, not analyse_eq's EZ / EM.
 *
 * Per chain c and event e, v = (x, y, z, t) of each used model: ref[c][k][e] = the chain's first used value, d = (double)v -
 * ref, sum[c][k][e] += d_k, cross[c][p][e] += d_i d_j over the pairs p = xx xy xz xt yy yz yt zz zt tt (round to nearest, no
 * contraction), n_models[c] += 1.  Each (chain, event) is summed in record order: the accumulators are a function of the
 * chain's records.  Histograms of x, y and z over the box the sampler keeps hypocentres in (lo = grid x0 / y0 / z0, hi =
 * lo + (n - 1) h), bin width w = bin_km: n_bins[a] = (int)((hi - lo) / w) + 1, a value goes to bin (int)((v - lo) / w)
 * (float arithmetic) clamped to [0, n_bins[a] - 1]; a value outside [lo, hi] is also counted in outside[e][a].
 * Layout: hist [n_events][n_bins[0] + n_bins[1] + n_bins[2]] (int32, x bins then y then z), outside [n_events][3] (int32),
 * ref and sum [n_chains][4][n_events], cross [n_chains][10][n_events] (double), n_models [n_chains] (int64).  Memory:
 * 18 doubles per (chain, event) + 8 bytes per chain + 4 (sum n_bins + 3) bytes per event.
 *
 * Summary: N = sum_c n_c; mean = sum_c (n_c ref_c + S_c) / N; with m_c = ref_c + S_c / n_c and W_c[ij] = C_c[ij] -
 * S_c[i] S_c[j] / n_c, cov = (sum_c W_c + sum_c n_c (m_c - mean)(m_c - mean)^T) / (N - 1) (chains with n_c = 0 add
 * nothing).  Quantiles of x, y, z at p = 0.025 0.16 0.5 0.84 0.975: target = p N, j = the smallest bin whose cumulative
 * count cum_j >= target, value = lo + w (j + (target - cum_{j-1}) / count_j).  Mode: the centre lo + (j + 0.5) w of the
 * fullest bin (the lowest index on a tie).  Error ellipsoid from the 3 x 3 (x, y, z) block: cyclic Jacobi in double,
 * axes = sqrt(eigenvalue) in descending order (1 sigma; a negative rounding residue gives 0), axis_dir[e][k] = the unit
 * vector (x, y, z) of axis k, signed so that v_z >= 0, or v_y >= 0 when v_z == 0, or v_x >= 0 when both are 0.  For a
 * confidence level P multiply the axes by sqrt(chi2_3(P)) (e.g. 2.796 for 95 %).  N = 0: everything NaN; N = 1: cov,
 * axes and axis_dir NaN.
 *
 * mq_hypo_begin allocates and zeroes the accumulators (again = restart), before or after mq_init_chains; MQ_ERR_ARG for
 * bin_km <= 0, more than 2^20 bins on an axis or a negative burn_in.  mq_hypo_chains copies the accumulators out.
 * mq_hypo_summary computes the summary on the device (fixed-order reductions, no floating-point atomics: the same
 * accumulators give the same bits): mean [n_events][4], cov [n_events][4][4], quant [n_events][3][5], mode [n_events][3],
 * axes [n_events][3], axis_dir [n_events][3][3], *n_models = N.  Any output pointer may be NULL.  With collective != 0 and
 * a communicator (mq_comm_init) the sums are all-reduced over the ranks in two rounds and the histograms as int32, and
 * every rank gets the job-wide numbers; without one, collective is ignored (outside stays per handle: mq_hypo_chains).
 * It first reports a pending error of an earlier asynchronous call.  Both return MQ_ERR_STATE before mq_hypo_begin.  The
 * accumulators are part of a saved state (MQ_STATE_HYPO). */
typedef struct mq_hypo_dims { int32_t n_events, n_bins[3]; float bin_km, lo[3]; } mq_hypo_dims;
int mq_hypo_begin(mq_handle* h, float bin_km, int64_t burn_in, mq_hypo_dims* dims);
int mq_hypo_chains(mq_handle* h, int32_t* hist, int32_t* outside, double* ref, double* sum, double* cross, int64_t* n_models);
int mq_hypo_summary(mq_handle* h, int collective, double* mean, double* cov, double* quant, double* mode, double* axes,
                    double* axis_dir, int64_t* n_models);

/* NCCL communicator of the job (one rank per handle).  Rank 0 calls mq_comm_unique_id and hands the 128 bytes to the
 * other ranks by whatever means the host has (torch.distributed broadcast, a file, MPI); every rank then calls
 * mq_comm_init.  libnccl is bound at run time; MQ_ERR_UNSUPPORTED when it is absent. */
#define MQ_COMM_ID_BYTES 128
int mq_comm_unique_id(uint8_t* id);
int mq_comm_init(mq_handle* h, const uint8_t* id, int rank, int world);
int mq_comm_destroy(mq_handle* h);

/* Optional parallel tempering (not reference behaviour): chain c samples prior x likelihood^beta[c]; beta == 1 is the
 * reference's chain.  mq_temper_swap proposes one round of swaps between neighbouring chains of the global numbering
 * (pairs (2k+p, 2k+1+p), p = round & 1): one all-gather of (log-likelihood, beta) per chain, identical decisions on
 * every rank from a shared counter-based stream keyed by (seed, round, pair), temperatures are swapped, states stay.
 * Works without a communicator (single GPU).  *n_swapped counts accepted swaps whose lower chain is on this rank. */
int mq_set_beta(mq_handle* h, const float* beta);
int mq_get_beta(mq_handle* h, float* beta);
int mq_temper_swap(mq_handle* h, int64_t round, int32_t* n_swapped);

/* ===== checkpoint and resume =================================================================================
 * Sampler state of every chain of the handle: what mq_step needs to continue each chain exactly where it is -- the
 * current model, hypocentres, origin times, station corrections, sigmas, per-event class sums, likelihood, counters, the
 * random-stream position (Philox counter) and LVZ switch of every chain, its best model so far, the posterior and
 * diagnostics accumulators and temperatures when they are on, the seed and the chain offset.  A handle that loads a state continues
 * every chain with the same proposals, decisions and records as the handle that saved it, bit for bit.
 *
 * mq_state_size: *bytes = the size of a state of this handle as it is now (the posterior and temperatures count only when
 *   they are on).
 * mq_state_save: writes the state into buf[0, cap), *bytes (may be NULL) = its size.  It first reports a pending error of
 *   an earlier asynchronous call.  MQ_ERR_STATE before there is a sampler state (mq_init_chains, or mq_set_models and a
 *   first mq_step) and while decimated records wait in the ring (records are not state: drain first, so that a resumed run
 *   never delivers a record twice); MQ_ERR_BUSY while a drain batch is in flight (mq_drain_begin .. mq_batch_release);
 *   MQ_ERR_ARG when cap is too small.
 * mq_state_load: replaces the sampler state of the handle -- fresh (no mq_init_chains) or one that has stepped -- by a saved
 *   one.  The state's seed, chain offset, posterior setting and temperatures replace the handle's; records still in the
 *   handle's ring are discarded.  A state that does not fit the handle -- other chain count or sizes, a configuration or
 *   pick set with another checksum (mq_create's inputs), another format version, a bad trailing checksum (truncated or
 *   damaged) -- is refused with MQ_ERR_ARG before anything on the device changes: the handle stays as it was.  The
 *   travel-time tables are not in the state; they are rebuilt, and their hashes compared with the saved ones: a table
 *   that differs (a library whose eikonal results differ) gives MQ_ERR_STATE, mq_last_error() names the first chain and
 *   phase, and the handle has no usable state until the next mq_state_load / mq_init_chains / mq_set_models.  A state
 *   saved with reciprocal tables (MQ_STATE_RECIPROCAL) loads only into a handle set to MQ_TABLES_RECIPROCAL, a state
 *   without the flag only into a parity handle; anything else is refused with MQ_ERR_ARG before the device changes.
 *
 * Layout (native little-endian): an mq_state_header, n_sections mq_state_section entries, the sections at their offsets
 * (8-byte aligned, zero padding), and a trailing uint64 checksum of every byte before it.  Checksums are sum64: starting
 * from h = 0x9E3779B97F4A7C15, for every 64-bit little-endian word w of the data (the last one zero-padded),
 * h = (h ^ w) * 0x100000001B3 and then h ^= h >> 32.  config_sum is sum64 of the mq_config with the bytes after each
 * string's NUL zeroed; picks_sum chains sum64 over (n_events, n_picks, n_stations), ev_off, n_p, st_id, x, y, z, t, cls,
 * (reftime != NULL, fix != NULL) and the arrays reftime and fix when present.  Sections: MQ_STATE_SEC_CHAINS = one record
 * per chain (layout given by the format version), MQ_STATE_SEC_TABLES = uint64 hash per (chain, phase P/S) of the stored
 * receiver rows, MQ_STATE_SEC_POSTERIOR = the int32 then (8-byte aligned) double accumulators of mq_posterior_begin,
 * MQ_STATE_SEC_BETA = float beta per chain, MQ_STATE_SEC_DIAG = the diagnostics' own parameters (int64 burn_in, int32
 * n_batches, int32 n_quantities), then ref, sum, sumsq (double), n_models (int64), batch_len and full_batches (int32) as
 * mq_diag_chains lays them out.  A state without diagnostics has no such flag or section: its layout does not depend on
 * whether the library knows them.  Loading replaces the handle's diagnostics, or frees them when the state has none; a
 * diagnostics section of another quantity count or a bad n_batches is refused with MQ_ERR_ARG.  MQ_STATE_SEC_HYPO =
 * the hypocentre accumulators' own parameters (int64 burn_in, float bin_km, int32 n_bins[3]), then hist and outside
 * (int32), zero padding to 8 bytes, ref, sum, cross (double) and n_models (int64) as mq_hypo_chains lays them out; the
 * same rules hold (flag MQ_STATE_HYPO, none: freed, a section whose bin width or bin counts do not fit: MQ_ERR_ARG). */
#define MQ_STATE_MAGIC "MQSTATE"
#define MQ_STATE_FORMAT 1
#define MQ_STATE_POSTERIOR 1u    /* flags */
#define MQ_STATE_BETA 2u
#define MQ_STATE_TABLES 4u       /* table hashes present (no tables exist with eikonal == 0 or aflag == 1) */
#define MQ_STATE_DIAG 8u         /* diagnostics accumulators present (mq_diag_begin) */
#define MQ_STATE_RECIPROCAL 16u  /* saved from a handle with reciprocal tables (mq_set_tables); set only with MQ_STATE_TABLES */
#define MQ_STATE_HYPO 32u        /* hypocentre accumulators present (mq_hypo_begin) */
#define MQ_STATE_SEC_CHAINS 1u
#define MQ_STATE_SEC_TABLES 2u
#define MQ_STATE_SEC_POSTERIOR 3u
#define MQ_STATE_SEC_BETA 4u
#define MQ_STATE_SEC_DIAG 5u
#define MQ_STATE_SEC_HYPO 6u
typedef struct mq_state_header {
    char magic[8];             /* MQ_STATE_MAGIC */
    uint32_t format;           /* MQ_STATE_FORMAT */
    uint32_t header_bytes;     /* sizeof(mq_state_header) */
    char version[48];          /* mq_version() of the library that saved it */
    int32_t n_chains, max_dim, n_events, n_stations, n_picks, nz, nxmod, n_rows;
    uint64_t seed;
    int64_t chain_offset;
    uint32_t flags;            /* MQ_STATE_POSTERIOR | MQ_STATE_BETA | MQ_STATE_TABLES | MQ_STATE_DIAG | MQ_STATE_RECIPROCAL | MQ_STATE_HYPO */
    uint32_t n_sections;
    float post_dv, post_dvpvs; /* mq_posterior_begin's arguments and the histogram sizes (0 when off) */
    int32_t post_ndv, post_ndvpvs;
    int64_t post_burn_in;
    uint64_t config_sum, picks_sum;
} mq_state_header;
typedef struct mq_state_section { uint32_t id, reserved; uint64_t offset, bytes; } mq_state_section;   /* offset from the blob's start */
int mq_state_size(mq_handle* h, uint64_t* bytes);
int mq_state_save(mq_handle* h, void* buf, uint64_t cap, uint64_t* bytes);
int mq_state_load(mq_handle* h, const void* buf, uint64_t bytes);

/* Measurement aid for bench.py: with enable != 0 every eikonal launch is bracketed by CUDA events on
 * the handle's stream.  Returns the time and number of launches accumulated since the previous call
 * (and restarts the accumulation); solves_per_full_launch = 2 * n_chains * nz (2 * n_chains * n_rows with reciprocal
 * tables), the number of solves one launch performs when every chain rebuilds both tables. */
int mq_profile(mq_handle* h, int enable, double* eikonal_ms, int64_t* eikonal_launches,
               int64_t* solves_per_full_launch);

/* Which eikonal kernel the launches counted by the last mq_profile call took: launches[k] / ms[k], k = 0 generic
 * (time field in global memory), 1 fused (one warp per CTA, shared memory), 2 pipelined (shared-memory box phase +
 * tensor-memory march), 3 fine-grid (planes that do not fit a shared-memory slice); both arrays hold MQ_EIK_KERNELS
 * entries.  mq_eikonal_kernel_name(k) is the kernel's symbol name as ncu prints it. */
#define MQ_EIK_KERNELS 4
int mq_profile_kernels(mq_handle* h, int64_t* launches, double* ms);
const char* mq_eikonal_kernel_name(int k);
/* The same accumulation for the lookup / residual kernel (misfit_kernel): launches and their summed device time. */
int mq_profile_misfit(mq_handle* h, int64_t* launches, double* ms);

/* CUDA-event stopwatch on the handle's stream: stop = 0 records the start of `slot` (0..15), stop = 1 records
 * the end, waits for it and returns the device time between the two in *elapsed_ms. */
int mq_timer(mq_handle* h, int slot, int stop, double* elapsed_ms);

#ifdef __cplusplus
}
#endif
#endif /* MCMCEQ_B200_H */
