/* oracle/pl_eikonal.c -- TEST INFRASTRUCTURE ONLY (CPU oracle).
 *
 * Re-entrant restatement of the Podvin & Lecomte (1991) expanding-box
 * finite-difference eikonal scheme as implemented by the reference
 * (src/time_2d.c).  Function-by-function map:
 *
 *   pl_time_2d        <- time_2d            src/time_2d.c:301-367
 *   grid_prepare      <- pre_init           src/time_2d.c:440-499
 *   seed_source       <- init_point         src/time_2d.c:503-717
 *   seed_cells/cell   <- init_nearest/init_cell/init_cellh   :724-802
 *   seed_refined      <- recursive_init     src/time_2d.c:806-917
 *   expand_box        <- propagate_point    src/time_2d.c:921-955
 *   sweep_line        <- y_side AND x_side  src/time_2d.c:959-1147, 1186-1373
 *   push_headwave     <- send_y_headwave / send_x_headwave   :1157, :1377
 *
 * The reference keeps its state in file-scope statics and has two textual
 * copies of the side sweep (one per axis); here the state is a context struct
 * and one strided sweep serves both axes.  Every floating-point expression
 * keeps the reference's operand types (float products, double sqrt and
 * M_SQRT2 terms rounded to float on assignment) so that results are
 * bit-identical; tests/test_oracle_pin.py checks exactly that against the
 * compiled reference (oracle/_ref).  Build with -ffp-contract=off.
 *
 * Not restated: the "multiple source" mode (source outside the grid, times
 * given on input) -- mcmc_eq never uses it (src/misfit.c:274-278).
 */
#include "pl_eikonal.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#ifndef M_SQRT2
#define M_SQRT2 1.41421356237309504880
#endif

#define PL_HUGE 0.499e+19f
#define PL_FUZZ 1.2e-07
#define PL_INIT_MIN 10
#define PL_FINE_MAX (4 * PL_INIT_MIN + 3)

typedef struct {
    int nx, ny;      /* nodes per axis                                   */
    int mx, my;      /* cells per axis (last cell row / column are dummy) */
    const float *hs; /* slowness*spacing per cell, x-major                */
    float *t;        /* node times, x-major                               */
    float fxs, fys;  /* source position (node units)                      */
    int xs, ys;      /* nearest node                                      */
    int at_node;
    int level;       /* 0 = caller's grid, 1 = refined grid round source  */
    float eps;
    int X0, X1, Y0, Y1; /* inclusive bounds of the timed box              */
    int rev_depth;      /* nesting of head-wave reverse propagation       */
    int side_limit;     /* line at which reverse propagation must stop    */
    pl_stats *st;
} grid_t;

static inline float fminf_ref(float a, float b) { return (a < b) ? a : b; }

/* ---- strided access: axis 0 walks along y on a fixed x (reference y_side),
 *      axis 1 walks along x on a fixed y (reference x_side) ---------------- */
static inline size_t at(const grid_t *g, int axis, int line, int k)
{
    return axis == 0 ? (size_t)line * g->ny + k : (size_t)k * g->ny + line;
}
#define TT(line, k) g->t[at(g, axis, (line), (k))]
#define SS(line, k) g->hs[at(g, axis, (line), (k))]

/* reference send_y_headwave/send_x_headwave, src/time_2d.c:1157-1182,1377-1402 */
static void push_headwave(grid_t *g, int axis, int from, int to, int line, int strip, int far)
{
    int k;
    float now, lo, est;
    if (from < to) {
        for (k = from; k < to; k++) {
            now = SS(strip, k);
            lo = (far < 0) ? now : fminf_ref(now, SS(far, k));
            if ((est = TT(line, k) + lo) < TT(line, k + 1)) TT(line, k + 1) = est;
        }
    } else {
        for (k = from; k > to; k--) {
            now = SS(strip, k - 1);
            lo = (far < 0) ? now : fminf_ref(now, SS(far, k - 1));
            if ((est = TT(line, k) + lo) < TT(line, k - 1)) TT(line, k - 1) = est;
        }
    }
}

/* One side of the box: times on `line` from the already timed line
 * `line-future`, between kb and ke inclusive.  Returns the number of stencil
 * adoptions (the reference's `updated`).  src/time_2d.c:959-1147 / 1186-1373. */
static int sweep_line(grid_t *g, int axis, int line, int future, int kb, int ke)
{
    const int past = line - future;
    const int strip = (future == 1) ? past : line; /* cell line between past and current */
    const int far = strip + future;                /* cell line beyond the current line  */
    const int across = (axis == 0) ? g->mx : g->my;
    int k, kmin, d, updated = 0, longhead = 0, alert;
    float hs0, hs1, hs2, est, dt;

    if (g->rev_depth == 0) g->side_limit = line + future;
    if (g->st) {
        if (axis == 0) g->st->col_sweeps++; else g->st->row_sweeps++;
        if (g->rev_depth) g->st->reverse_sweeps++;
    }

    for (k = kb; k <= ke;) {
        /* next local minimum of the past line (:990 / :1217) */
        while (k < ke && TT(past, k + 1) < TT(past, k)) k++;
        kmin = k;

        /* 1-D transmission in front of the minimum (:994-1000 / :1221-1227) */
        hs1 = SS(strip, k);
        hs0 = (k == 0) ? PL_INFINITY : SS(strip, k - 1);
        if ((est = TT(past, k) + fminf_ref(hs0, hs1)) < TT(line, k)) {
            TT(line, k) = est;
            updated++;
        }

        /* walk away from the minimum: first towards kb (d=-1), then towards ke (d=+1) */
        for (d = -1; d <= 1; d += 2) {
            if (d == 1 && kmin == ke) break;
            k = kmin + d;
            alert = 0;
            while ((d < 0 ? k >= kb : k <= ke) && (dt = TT(past, k) - TT(past, k - d)) >= 0.0) {
                const int n = k - d;               /* neighbour towards the minimum        */
                const int c0 = (d > 0) ? k - 1 : k; /* cell between k and n                */
                const int c1 = (d > 0) ? k : k - 1; /* next cell away from the minimum     */
                hs0 = SS(strip, c0);
                /* plane wave through the past side (:1007-1011) */
                if (dt < hs0 / M_SQRT2 && (est = TT(past, k) + sqrt(hs0 * hs0 - dt * dt)) < TT(line, k)) {
                    TT(line, k) = est;
                    updated++;
                }
                /* plane wave through the lateral side (:1012-1017) */
                dt = TT(line, n) - TT(past, n);
                if (dt >= 0.0 && dt < hs0 / M_SQRT2 &&
                    (est = TT(line, n) + sqrt(hs0 * hs0 - dt * dt)) < TT(line, k)) {
                    TT(line, k) = est;
                    updated++;
                }
                /* 1-D transmission towards the future (:1018-1024, :1080-1084) */
                if (d > 0 || k != 0) {
                    hs1 = SS(strip, c1);
                    if ((est = TT(past, k) + hs1) < TT(line, k)) {
                        TT(line, k) = est;
                        updated++;
                    }
                }
                /* corner diffraction (:1025-1028) */
                if ((est = TT(past, n) + hs0 * M_SQRT2) < TT(line, k)) {
                    TT(line, k) = est;
                    updated++;
                }
                /* head wave along the current line (:1029-1059) */
                if (far >= 0) {
                    hs2 = SS(far, c0);
                    if (hs2 < hs0) {
                        est = TT(line, n) + hs2;
                        dt = TT(line, k) - est;
                        if (dt > PL_FUZZ * TT(line, k)) {
                            TT(line, k) = est;
                            updated++;
                            if (!alert) {
                                longhead++;
                                push_headwave(g, axis, k, (d < 0) ? kb : ke, line, strip, far);
                                alert = 1;
                            }
                        } else {
                            alert = 0;
                            est = TT(line, k) + hs2;
                            dt = TT(line, n) - est;
                            if (dt > PL_FUZZ * TT(line, n)) {
                                TT(line, n) = est;
                                updated++;
                                push_headwave(g, axis, n, (d < 0) ? ke : kb, line, strip, far);
                                longhead++;
                            }
                        }
                    }
                }
                k += d;
            }
        }
        if (kmin == ke) break;
    }

    /* a head wave ran along this line: re-time the lines behind it (:1128-1143) */
    if (longhead) {
        int l;
        if (g->st) g->st->headwaves += longhead;
        g->rev_depth++;
        if (g->st && g->rev_depth > g->st->max_rev_depth) g->st->max_rev_depth = g->rev_depth;
        for (l = past; l != g->side_limit; l -= future) {
            if (l < 0 || l > across) break;
            if (sweep_line(g, axis, l, -future, kb, ke) == 0) break;
        }
        g->rev_depth--;
    }
    return updated;
}

/* reference propagate_point, src/time_2d.c:921-955 */
static void expand_box(grid_t *g)
{
    int moved;
    do {
        moved = 0;
        if (g->X0 > 0) { g->X0--; sweep_line(g, 0, g->X0, -1, g->Y0, g->Y1); moved++; }
        if (g->Y0 > 0) { g->Y0--; sweep_line(g, 1, g->Y0, -1, g->X0, g->X1); moved++; }
        if (g->X1 < g->mx) { g->X1++; sweep_line(g, 0, g->X1, 1, g->Y0, g->Y1); moved++; }
        if (g->Y1 < g->my) { g->Y1++; sweep_line(g, 1, g->Y1, 1, g->X0, g->X1); moved++; }
    } while (moved);
}

/* reference init_cellh, src/time_2d.c:791-802 */
static float head_in_cell(float vh, float vv, float hsc, float hsn)
{
    float hsd;
    hsd = sqrt(hsc * hsc - hsn * hsn);
    if (vh * hsd > vv * hsn) return vh * hsn + vv * hsd;
    return PL_INFINITY;
}

/* reference init_cell, src/time_2d.c:758-789 (x,y: cell; dx,dy: source offset from its corner) */
static void seed_cell(grid_t *g, float dx, float dy, int x, int y)
{
    const int ny = g->ny;
    float *t = g->t;
    const float *hs = g->hs;
    float hs0, hs1, est;
#define T2(a, b) t[(size_t)(a) * ny + (b)]
#define S2(a, b) hs[(size_t)(a) * ny + (b)]
    hs0 = S2(x, y);
    if ((est = hs0 * sqrt(dx * dx + dy * dy)) < T2(x, y)) T2(x, y) = est;
    if ((est = hs0 * sqrt((1.0 - dx) * (1.0 - dx) + dy * dy)) < T2(x + 1, y)) T2(x + 1, y) = est;
    if ((est = hs0 * sqrt(dx * dx + (1.0 - dy) * (1.0 - dy))) < T2(x, y + 1)) T2(x, y + 1) = est;
    if ((est = hs0 * sqrt((1.0 - dx) * (1.0 - dx) + (1.0 - dy) * (1.0 - dy))) < T2(x + 1, y + 1))
        T2(x + 1, y + 1) = est;
    if (x && (hs1 = S2(x - 1, y)) < hs0) {
        if ((est = head_in_cell(dx, dy, hs0, hs1)) < T2(x, y)) T2(x, y) = est;
        if ((est = head_in_cell(dx, 1.0 - dy, hs0, hs1)) < T2(x, y + 1)) T2(x, y + 1) = est;
    }
    if (y && (hs1 = S2(x, y - 1)) < hs0) {
        if ((est = head_in_cell(dy, dx, hs0, hs1)) < T2(x, y)) T2(x, y) = est;
        if ((est = head_in_cell(dy, 1.0 - dx, hs0, hs1)) < T2(x + 1, y)) T2(x + 1, y) = est;
    }
    /* the reference tests x against nmesh_y here (src/time_2d.c:781); kept as is */
    if (x < g->my - 1 && (hs1 = S2(x + 1, y)) < hs0) {
        if ((est = head_in_cell(1.0 - dx, dy, hs0, hs1)) < T2(x + 1, y)) T2(x + 1, y) = est;
        if ((est = head_in_cell(1.0 - dx, 1.0 - dy, hs0, hs1)) < T2(x + 1, y + 1)) T2(x + 1, y + 1) = est;
    }
    if (y < g->my - 1 && (hs1 = S2(x, y + 1)) < hs0) {
        if ((est = head_in_cell(1.0 - dy, dx, hs0, hs1)) < T2(x, y + 1)) T2(x, y + 1) = est;
        if ((est = head_in_cell(1.0 - dy, 1.0 - dx, hs0, hs1)) < T2(x + 1, y + 1)) T2(x + 1, y + 1) = est;
    }
#undef T2
#undef S2
}

/* reference init_nearest, src/time_2d.c:724-756 */
static void seed_cells(grid_t *g)
{
    const int xs = g->xs, ys = g->ys;
    if (g->st) g->st->nearest_init++;
    if (g->at_node) {
        if (xs < g->mx && ys < g->my) seed_cell(g, 0.f, 0.f, xs, ys);
        if (xs && ys < g->my) seed_cell(g, 1.f, 0.f, xs - 1, ys);
        if (xs < g->mx && ys) seed_cell(g, 0.f, 1.f, xs, ys - 1);
        if (xs && ys) seed_cell(g, 1.f, 1.f, xs - 1, ys - 1);
        return;
    }
    {
        int x = (g->fxs < xs) ? xs - 1 : xs;
        int y = (g->fys < ys) ? ys - 1 : ys;
        float dx = g->fxs - x, dy = g->fys - y;
        if (xs == g->fxs) {
            seed_cell(g, 0.f, dy, x, y);
            if (x) seed_cell(g, 1.f, dy, x - 1, y);
        } else if (ys == g->fys) {
            seed_cell(g, dx, 0.f, x, y);
            if (y) seed_cell(g, dx, 1.f, x, y - 1);
        } else {
            seed_cell(g, dx, dy, x, y);
        }
    }
}

static int solve_grid(grid_t *g);

/* Geometry of the half-spacing grid along one axis (src/time_2d.c:844-864):
 * n fine nodes, fine source node src, coarse cell c0 under fine cell 0, and
 * whether fine cell 0 is the second half of its coarse cell (half=1). */
static void refine_axis(int s_coarse, int n_coarse, int *n, int *src, int *c0, int *half)
{
    int d;
    *n = PL_FINE_MAX;
    *src = 2 * PL_INIT_MIN + 1;
    *half = 1;
    *c0 = s_coarse - PL_INIT_MIN - 1;
    if ((d = PL_INIT_MIN - s_coarse) >= 0) {
        *c0 += d + 1;
        d = 1 + 2 * d;
        *n -= d;
        *src -= d;
        *half = 0;
    }
    if ((d = s_coarse + PL_INIT_MIN - n_coarse + 1) >= 0) *n -= 1 + 2 * d;
}

/* reference recursive_init, src/time_2d.c:806-917 */
static int seed_refined(grid_t *g)
{
    float HS[PL_FINE_MAX * PL_FINE_MAX], T[PL_FINE_MAX * PL_FINE_MAX];
    grid_t f;
    int nxf, nyf, xsf, ysf, i0, j0, hx, hy, ii, jj, n, rc;

    if (g->st) g->st->recursive_init++;
    for (n = 0; n < PL_FINE_MAX * PL_FINE_MAX; n++) HS[n] = T[n] = PL_INFINITY;
    refine_axis(g->xs, g->nx, &nxf, &xsf, &i0, &hx);
    refine_axis(g->ys, g->ny, &nyf, &ysf, &j0, &hy);
    for (n = 0, ii = 0; ii < nxf; ii++) {
        const int i = i0 + (hx ? (ii + 1) / 2 : ii / 2);
        for (jj = 0; jj < nyf; jj++, n++) {
            const int j = j0 + (hy ? (jj + 1) / 2 : jj / 2);
            HS[n] = 0.5 * g->hs[(size_t)i * g->ny + j]; /* no smoothing */
        }
    }

    memset(&f, 0, sizeof f);
    f.nx = nxf;
    f.ny = nyf;
    f.hs = HS;
    f.t = T;
    f.fxs = xsf + 2.0 * (g->fxs - g->xs);
    f.fys = ysf + 2.0 * (g->fys - g->ys);
    f.level = g->level + 1;
    f.eps = g->eps;
    f.st = g->st;
    rc = solve_grid(&f);
    if (rc != PL_OK) return PL_ERR_RECURS;

    /* every second fine node is a coarse node (:887-890) */
    {
        int i, j;
        for (i = i0 + hx, ii = hx; ii < nxf; ii += 2, i++)
            for (j = j0 + hy, jj = hy; jj < nyf; jj += 2, j++)
                g->t[(size_t)i * g->ny + j] = T[ii * nyf + jj];
    }
    return PL_OK;
}

/* reference init_point (single point source branch), src/time_2d.c:503-717 */
static int seed_source(grid_t *g)
{
    const int mx = g->mx, my = g->my, ny = g->ny;
    int x, y, xsc, ysc, tried;
    int failW = 0, failE = 0, failN = 0, failS = 0;
    float hs0, tol, sq;

    if (!(g->fxs >= 0.0 && g->fxs <= mx && g->fys >= 0.0 && g->fys <= my)) return PL_ERR_SOURCE;
    if (g->level == 0) {
        size_t i, n = (size_t)g->nx * g->ny;
        if (g->eps < 0.0 || g->eps > 1.0) return PL_ERR_EPS;
        for (i = 0; i < n; i++) g->t[i] = PL_INFINITY;
    }
    g->xs = (int)floor(g->fxs + 0.5);
    g->ys = (int)floor(g->fys + 0.5);
    g->at_node = (g->xs == g->fxs && g->ys == g->fys);

    if (g->at_node) {
        xsc = (g->xs == mx) ? g->xs - 1 : g->xs;
        ysc = (g->ys == my) ? g->ys - 1 : g->ys;
    } else {
        xsc = (g->fxs < g->xs) ? g->xs - 1 : g->xs;
        ysc = (g->fys < g->ys) ? g->ys - 1 : g->ys;
    }
    hs0 = g->hs[(size_t)xsc * ny + ysc];

    /* largest quasi-square box of cells with slowness within eps of hs0 (:594-644) */
    tol = hs0 * g->eps;
    g->X0 = g->X1 = xsc;
    g->Y0 = g->Y1 = ysc;
#define DIFFERS(a, b) (fabs(g->hs[(size_t)(a) * ny + (b)] - hs0) > tol)
    do {
        tried = 0;
        if (g->X0 && !failW) {
            tried++;
            x = --g->X0;
            for (y = g->Y0; y <= g->Y1 && !failW; y++) if (DIFFERS(x, y)) failW = 1;
            if (failW) g->X0++;
        }
        if (g->Y0 && !failN) {
            tried++;
            y = --g->Y0;
            for (x = g->X0; x <= g->X1 && !failN; x++) if (DIFFERS(x, y)) failN = 1;
            if (failN) g->Y0++;
        }
        if (g->X1 < mx - 1 && !failE) {
            tried++;
            x = ++g->X1;
            for (y = g->Y0; y <= g->Y1 && !failE; y++) if (DIFFERS(x, y)) failE = 1;
            if (failE) g->X1--;
        }
        if (g->Y1 < my - 1 && !failS) {
            tried++;
            y = ++g->Y1;
            for (x = g->X0; x <= g->X1 && !failS; x++) if (DIFFERS(x, y)) failS = 1;
            if (failS) g->Y1--;
        }
        /* stop at the first round in which any side met a heterogeneity (:642) */
        if (tried && (failW + failE + failN + failS)) tried = 0;
    } while (tried);
#undef DIFFERS
    /* cells -> nodes, then keep heterogeneous interfaces out of the exact zone (:645-663) */
    g->X1++;
    g->Y1++;
    if (failW) g->X0++;
    if (failN) g->Y0++;
    if (failE) g->X1--;
    if (failS) g->Y1--;
    if (g->X0 > g->fxs || g->X1 < g->fxs || g->Y0 > g->fys || g->Y1 < g->fys) {
        g->X0 = xsc;
        g->Y0 = ysc;
        g->X1 = xsc + 1;
        g->Y1 = ysc + 1;
    }

    if (g->level >= 1 ||
        ((g->X0 == 0 || (g->xs - g->X0) >= PL_INIT_MIN) && (g->Y0 == 0 || (g->ys - g->Y0) >= PL_INIT_MIN) &&
         (g->X1 == mx || (g->X1 - g->xs) >= PL_INIT_MIN) && (g->Y1 == my || (g->Y1 - g->ys) >= PL_INIT_MIN))) {
        if ((g->X1 - g->X0) * (g->Y1 - g->Y0) == 1) {
            seed_cells(g);
        } else {
            if (g->st) g->st->box_init++;
            for (x = g->X0; x <= g->X1; x++)
                for (y = g->Y0; y <= g->Y1; y++) {
                    sq = (x - g->fxs) * (x - g->fxs) + (y - g->fys) * (y - g->fys);
                    g->t[(size_t)x * ny + y] = hs0 * sqrt(sq);
                }
        }
        return PL_OK;
    }
    {
        int rc = seed_refined(g);
        if (rc != PL_OK) return rc;
    }
    g->X0 = (g->xs - PL_INIT_MIN > 0) ? g->xs - PL_INIT_MIN : 0;
    g->Y0 = (g->ys - PL_INIT_MIN > 0) ? g->ys - PL_INIT_MIN : 0;
    g->X1 = (g->xs + PL_INIT_MIN < mx) ? g->xs + PL_INIT_MIN : mx;
    g->Y1 = (g->ys + PL_INIT_MIN < my) ? g->ys + PL_INIT_MIN : my;
    return PL_OK;
}

static int solve_grid(grid_t *g)
{
    int rc;
    if (g->nx < 2 || g->ny < 2) return PL_ERR_DIM;
    g->mx = g->nx - 1;
    g->my = g->ny - 1;
    g->rev_depth = 0;
    rc = seed_source(g);
    if (rc == PL_OK) expand_box(g);
    return rc;
}

int pl_time_2d(const float *hs, float *t, int nx, int ny, float xs, float ys, float eps_init, pl_stats *stats)
{
    grid_t g;
    float *masked;
    int i, j, rc, err = PL_OK;

    if (nx < 2 || ny < 2) return PL_ERR_DIM;
    /* licit-value scan over the non-dummy cells, same visiting order and
     * last-writer-wins behaviour as src/time_2d.c:469-480 */
    for (i = 0; i < nx - 1; i++)
        for (j = 0; j < ny - 1 && err == PL_OK; j++) {
            if (hs[(size_t)i * ny + j] > PL_HUGE) err = PL_ERR_RANGE;
            if (hs[(size_t)i * ny + j] < 0.0) err = PL_ERR_PHYS;
        }
    if (err != PL_OK) return err;

    /* the reference masks the dummy row/column in place and restores them on
     * exit (:489-496, :359-360); a private copy gives the same solve */
    masked = (float *)malloc((size_t)nx * ny * sizeof(float));
    if (!masked) return PL_ERR_ALLOC;
    memcpy(masked, hs, (size_t)nx * ny * sizeof(float));
    for (i = 0; i < nx; i++) masked[(size_t)i * ny + (ny - 1)] = PL_INFINITY;
    for (j = 0; j < ny - 1; j++) masked[(size_t)(nx - 1) * ny + j] = PL_INFINITY;

    memset(&g, 0, sizeof g);
    g.nx = nx;
    g.ny = ny;
    g.hs = masked;
    g.t = t;
    g.fxs = xs;
    g.fys = ys;
    g.eps = eps_init;
    g.level = 0;
    g.st = stats;
    rc = solve_grid(&g);
    free(masked);
    return rc;
}
