/* oracle/pl_eikonal.h -- TEST INFRASTRUCTURE ONLY (CPU oracle).
 *
 * Re-entrant CPU restatement of the Podvin-Lecomte finite-difference eikonal
 * solver exactly as mcmc_eq calls it (reference: src/time_2d.c:301-1402,
 * prototype src/fdtimes.h:6-7).  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may link or call this; the
 * product library (mcmc_eq_b200/csrc) never does.
 *
 * Parity pin: tests/test_oracle_pin.py compares pl_time_2d() bit-for-bit with
 * the unmodified reference compiled into oracle/_ref/libmcmceq_ref.so, and
 * with the committed fixtures tests/golden/ that were generated from it.
 */
#ifndef ORACLE_PL_EIKONAL_H
#define ORACLE_PL_EIKONAL_H

#ifdef __cplusplus
extern "C" {
#endif

#define PL_INFINITY 0.500e+19f
#define PL_OK 0
#define PL_ERR_ALLOC (-3)
#define PL_ERR_RECURS (-4)
#define PL_ERR_EPS (-5)
#define PL_ERR_RANGE (-6)
#define PL_ERR_PHYS (-7)
#define PL_ERR_DIM (-8)
#define PL_ERR_SOURCE (-20) /* source outside the grid: "multiple source" mode is not on the hot path */

/* Event counters filled by pl_time_2d when stats != NULL (diagnostics used by
 * the tests to make sure the irregular branches are actually exercised). */
typedef struct {
    long col_sweeps;      /* sweeps along depth  (reference y_side) */
    long row_sweeps;      /* sweeps along distance (reference x_side) */
    long reverse_sweeps;  /* sweeps issued from a head-wave reverse propagation */
    long headwaves;       /* head-wave adoptions that raised reverse propagation */
    long recursive_init;  /* half-spacing re-discretised initialisations */
    long nearest_init;    /* minimal (<=4 cell) initialisations */
    long box_init;        /* analytic homogeneous-box initialisations */
    long max_rev_depth;   /* deepest nesting of head-wave reverse propagation (frames open at once) */
} pl_stats;

/* Same contract as the reference time_2d(): hs and t are [nx][ny] arrays,
 * x-major (index x*ny+y); hs holds slowness*spacing per cell (last row and
 * column are dummies); (xs,ys) is the source in node units.  Unlike the
 * reference the caller's hs array is never written to.  Returns 0 or a
 * negative PL_ERR_* code. */
int pl_time_2d(const float *hs, float *t, int nx, int ny, float xs, float ys,
               float eps_init, pl_stats *stats);

#ifdef __cplusplus
}
#endif
#endif
