// eik_core.cuh -- one-lane-per-solve Podvin-Lecomte eikonal, FP32, for the only
// call pattern on mcmc_eq's hot path:
//
//     time_2d(hs, t, nxmod, nz, xs = 0, ys = iz, eps = 0.001, 0)      (reference src/misfit.c:278)
//
// i.e. a depth-only medium (hs[x][y] = s[y], reference src/misfit.c:257-266) and a
// source that is a grid node on the left edge.  Behaviour follows reference
// src/time_2d.c:301-1402 (SURVEY.md Appendix A); the structure does not:
//   * state lives in a per-lane struct, never in statics, so thousands of solves run at once;
//   * one strided sweep serves rows and columns (the reference has two textual copies);
//   * the box never grows to the left (X0 == 0 for a left-edge source) and the
//     homogeneous-box search only ever tests one cell per row (depth-only medium);
//   * head-wave reverse propagation is an explicit per-lane stack, not recursion;
//   * all arithmetic is FP32 (the reference mixes float storage with double sqrt/M_SQRT2);
//     results agree to |dT| <= max(1e-4 s, 2e-6 T), see tests/test_eikonal_*.py.
//
// The file compiles for the device (nvcc) and for the host (g++), bit-identically
// (-fmad=false / -ffp-contract=off, explicit fmaf), so the tolerance can be studied
// against the oracle on CPU; the host build is test-only (tests/emu).
#pragma once
#include <math.h>
#include <stddef.h>

#ifdef __CUDACC__
#define EIK_HD __host__ __device__ __forceinline__
#define EIK_HD_NOINLINE __host__ __device__ __noinline__
#else
#define EIK_HD inline
#define EIK_HD_NOINLINE
#endif

namespace eik {

constexpr float kInf = 0.500e+19f;   // reference INFINITY_FD, src/time_2d.c:181
constexpr float kFuzz = 1.2e-07f;    // reference EPS_FUZZY,  src/time_2d.c:189
constexpr int kInitMin = 10;         // reference INIT_MIN,    src/time_2d.c:238
constexpr int kFineMax = 4 * kInitMin + 3;
constexpr float kSqrt2 = 1.41421356237309504880f;
constexpr float kRsqrt2 = 0.70710678118654752440f;
constexpr int kMaxReverseDepth = 12;

enum Status : int {
    kOk = 0,
    kErrRecurs = -4,
    kErrDim = -8,
    kErrReverseDepth = -30,  // head-wave reverse propagation nested deeper than kMaxReverseDepth
};

struct Counters {  // optional diagnostics, one per lane
    int col_sweeps, row_sweeps, reverse_sweeps, headwaves, recursive_init, nearest_init, box_init;
};

EIK_HD float fmin_ref(float a, float b) { return (a < b) ? a : b; }

// t + sqrt(r) rounded once, the way the reference's (float)(t + sqrt((double)r)) is
// (src/time_2d.c:1008): the correctly rounded sqrtf plus its first-order residual.
EIK_HD float add_sqrt(float t, float r)
{
    const float s = sqrtf(r);
#ifdef EIK_COMPENSATED
    if (s > 0.f) {
        const float e = fmaf(-s, s, r);       // r - s*s, exact
        const float c = e * (0.5f / s);       // sqrt(r) ~= s + c
        const float sum = t + s;
        const float err = (t - sum) + s;      // Fast2Sum tail (t >= s away from the source; harmless otherwise)
        return sum + (err + c);
    }
#endif
    return t + s;
}

// Coarse (caller's) medium: s[cy] for real cells, INFINITY on the dummy row and column
// that the reference masks for the duration of a top-level call (src/time_2d.c:489-496).
struct CoarseMedium {
    const float* s;   // nz values; s[my] is a dummy
    int sstride;      // element stride of s
    int mx, my;
    EIK_HD float operator()(int cx, int cy) const
    {
        return (cx >= mx || cy >= my) ? kInf : s[(size_t)cy * sstride];
    }
};

// Half-spacing medium of the re-discretised initialisation (src/time_2d.c:865-871):
// every coarse cell becomes 2x2 fine cells of half the slowness*spacing, no smoothing,
// and the fine grid's own dummy row/column carry real values (they are NOT masked).
struct FineMedium {
    CoarseMedium c;
    int j0, hy;   // coarse row under fine row 0; 1 when fine row 0 is the second half of its coarse cell
    EIK_HD float operator()(int cx, int cy) const { return 0.5f * c(cx >> 1, j0 + ((cy + hy) >> 1)); }
};

// Time field of one lane: node (x,y) lives at t[(x*ny + y)*ts]; ts = 32 interleaves the
// lanes of a warp so that lanes working on the same node touch one 128-byte line.
// View: what a sweep reads of a grid, handed to it by value.  Through a reference the struct
// would live in the caller's frame, and since a store to a node may alias it, every node
// access would re-read t, ny, ts and the medium from local memory.
template <class Medium>
struct View {
    float* t;
    int ts, ny;
    Medium S;
    EIK_HD float& T(int x, int y) const { return t[((size_t)x * ny + y) * ts]; }
};

template <class Medium>
struct Grid {
    float* t;
    int ts;
    int nx, ny, mx, my;
    Medium S;
    int ys;               // source node (0, ys)
    int X1, Y0, Y1;       // timed box, inclusive; X0 == 0 always
    int status;
    Counters* cnt;
    EIK_HD float& T(int x, int y) const { return t[((size_t)x * ny + y) * ts]; }
    EIK_HD View<Medium> view() const { return View<Medium>{t, ts, ny, S}; }
    EIK_HD void note(int st) { if (st != kOk) status = st; }
};

#define EIK_CNT(g, f) do { if ((g).cnt) (g).cnt->f++; } while (0)

// --- one line -------------------------------------------------------------------------
// AXIS 0: the line is a column x = `line`, k runs along depth   (reference y_side, :959-1147)
// AXIS 1: the line is a row    y = `line`, k runs along distance (reference x_side, :1186-1373)
template <int AXIS, class G>
EIK_HD float& node(const G& g, int line, int k) { return AXIS == 0 ? g.T(line, k) : g.T(k, line); }
template <int AXIS, class G>
EIK_HD float cell(const G& g, int line, int k) { return AXIS == 0 ? g.S(line, k) : g.S(k, line); }

template <int AXIS, class G>
EIK_HD void push_headwave(const G& g, int from, int to, int line, int strip, int far)
{   // reference send_y_headwave / send_x_headwave, src/time_2d.c:1157-1182, 1377-1402
    if (from < to) {
        for (int k = from; k < to; k++) {
            const float now = cell<AXIS>(g, strip, k);
            const float lo = (far < 0) ? now : fmin_ref(now, cell<AXIS>(g, far, k));
            const float est = node<AXIS>(g, line, k) + lo;
            if (est < node<AXIS>(g, line, k + 1)) node<AXIS>(g, line, k + 1) = est;
        }
    } else {
        for (int k = from; k > to; k--) {
            const float now = cell<AXIS>(g, strip, k - 1);
            const float lo = (far < 0) ? now : fmin_ref(now, cell<AXIS>(g, far, k - 1));
            const float est = node<AXIS>(g, line, k) + lo;
            if (est < node<AXIS>(g, line, k - 1)) node<AXIS>(g, line, k - 1) = est;
        }
    }
}

// Times on `line` from the timed line `line - future`, k in [kb, ke].  Returns the number of
// stencil adoptions; *longhead counts head waves that call for reverse propagation.
template <int AXIS, class G>
EIK_HD int walk_line(const G& g, int line, int future, int kb, int ke, int* longhead_out)
{
    const int past = line - future;
    const int strip = (future == 1) ? past : line;
    const int far = strip + future;
    int updated = 0, longhead = 0;

    for (int k = kb; k <= ke;) {
        // next local minimum of the past line
        float pk = node<AXIS>(g, past, k);
        while (k < ke) {
            const float pn = node<AXIS>(g, past, k + 1);
            if (!(pn < pk)) break;
            pk = pn;
            k++;
        }
        const int kmin = k;
        const float pmin = pk;
        {   // 1-D transmission in front of the minimum
            const float hs1 = cell<AXIS>(g, strip, k);
            const float hs0 = (k == 0) ? kInf : cell<AXIS>(g, strip, k - 1);
            const float est = pk + fmin_ref(hs0, hs1);
            if (est < node<AXIS>(g, line, k)) { node<AXIS>(g, line, k) = est; updated++; }
        }

        for (int d = -1; d <= 1; d += 2) {
            if (d == 1 && kmin == ke) break;
            k = kmin + d;
            int alert = 0;
            float pn = pmin;   // past-line time at the neighbour towards the minimum
            // current-line time at that neighbour; re-read because a backward head wave may
            // have been pushed over the minimum before the forward walk starts
            float cn = node<AXIS>(g, line, kmin);
            while (d < 0 ? k >= kb : k <= ke) {
                const float pk2 = node<AXIS>(g, past, k);
                float dt = pk2 - pn;
                if (!(dt >= 0.f)) break;
                const int n = k - d;
                const int c0 = (d > 0) ? k - 1 : k;
                const float hs0 = cell<AXIS>(g, strip, c0);
                const float lim = hs0 * kRsqrt2;
                const float hs0sq = hs0 * hs0;
                float c = node<AXIS>(g, line, k);
                float est;
                // plane wave through the past side
                if (dt < lim) {
                    est = add_sqrt(pk2, fmaf(-dt, dt, hs0sq));
                    if (est < c) { c = est; updated++; }
                }
                // plane wave through the lateral side (uses the value just computed at n)
                dt = cn - pn;
                if (dt >= 0.f && dt < lim) {
                    est = add_sqrt(cn, fmaf(-dt, dt, hs0sq));
                    if (est < c) { c = est; updated++; }
                }
                // 1-D transmission towards the future
                if (d > 0 || k != 0) {
                    const float hs1 = cell<AXIS>(g, strip, (d > 0) ? k : k - 1);
                    est = pk2 + hs1;
                    if (est < c) { c = est; updated++; }
                }
                // corner diffraction
                est = fmaf(hs0, kSqrt2, pn);
                if (est < c) { c = est; updated++; }
                // head wave along the current line
                if (far >= 0) {
                    const float hs2 = cell<AXIS>(g, far, c0);
                    if (hs2 < hs0) {
                        est = cn + hs2;
                        dt = c - est;
                        if (dt > kFuzz * c) {
                            c = est;
                            updated++;
                            if (!alert) {
                                longhead++;
                                node<AXIS>(g, line, k) = c;
                                push_headwave<AXIS>(g, k, (d < 0) ? kb : ke, line, strip, far);
                                alert = 1;
                            }
                        } else {
                            alert = 0;
                            est = c + hs2;
                            dt = cn - est;
                            if (dt > kFuzz * cn) {
                                node<AXIS>(g, line, n) = est;
                                updated++;
                                push_headwave<AXIS>(g, n, (d < 0) ? ke : kb, line, strip, far);
                                longhead++;
                            }
                        }
                    }
                }
                node<AXIS>(g, line, k) = c;
                pn = pk2;
                cn = c;
                k += d;
            }
        }
        if (kmin == ke) break;
    }
    *longhead_out = longhead;
    return updated;
}

// A side of the box plus, when a head wave ran along it, the reverse propagation of
// src/time_2d.c:1128-1143 / 1355-1369, unrolled into an explicit stack.  Recursively:
//     side(line, F): walk the line; if a head wave called for it,
//                    for l = line - F, line - 2F, ... (not side_limit, inside the grid): stop once side(l, -F) updates nothing
// `across`: the last line of this axis (mx for columns, my for rows).  Returns kOk or kErrReverseDepth.
// The stack holds one int per frame, in registers: frame f walks lines in the direction -F_f, where F_0 = future and
// F_{f+1} = -F_f (a frame is opened by a sweep of its parent's lines, whose future is -F_f), so only the frame's current
// line has to be kept; it lives in a shift register (lines[0] is the top), which unrolls to fixed indices, where an array
// indexed by the stack pointer would live in local memory.  Every frame is opened by a sweep that updated nodes (a head
// wave is an update), so a closed frame always tells its parent to go on.
template <int AXIS, class Medium>
EIK_HD_NOINLINE int sweep_line(const View<Medium> g, int across, int line, int future, int kb, int ke, Counters* cnt)
{
    int lines[kMaxReverseDepth];
#pragma unroll
    for (int i = 0; i < kMaxReverseDepth; i++) lines[i] = 0;
    int sp = 0, status = kOk;
    const int side_limit = line + future;
    int curL = line, curF = future;
    for (;;) {
        int lh = 0;
        const int upd = walk_line<AXIS>(g, curL, curF, kb, ke, &lh);
        if (cnt) {
            if (AXIS == 0) cnt->col_sweeps++; else cnt->row_sweeps++;
            if (sp) cnt->reverse_sweeps++;
            cnt->headwaves += lh;
        }
        if (lh && sp == kMaxReverseDepth) { status = kErrReverseDepth; lh = 0; }
        bool advance;   // move the top frame on to its next line (else: check the line it was just opened at)
        if (lh) {
#pragma unroll
            for (int i = kMaxReverseDepth - 1; i > 0; i--) lines[i] = lines[i - 1];
            lines[0] = curL - curF;
            sp++;
            advance = false;
        } else {
            if (sp == 0) return status;
            advance = true;
            if (upd == 0) {              // the re-timed line changed nothing: the frame is closed
#pragma unroll
                for (int i = 0; i < kMaxReverseDepth - 1; i++) lines[i] = lines[i + 1];
                if (--sp == 0) return status;
            }
        }
        for (;;) {
            const int F = (sp & 1) ? future : -future;   // F of the top frame, number sp - 1
            if (advance) lines[0] -= F;
            advance = true;
            const int l = lines[0];
            if (l == side_limit || l < 0 || l > across) {
#pragma unroll
                for (int i = 0; i < kMaxReverseDepth - 1; i++) lines[i] = lines[i + 1];
                if (--sp == 0) return status;
                continue;
            }
            curL = l;
            curF = -F;
            break;
        }
    }
}

// reference propagate_point, src/time_2d.c:921-955 (X0 == 0: the left side never moves)
template <class G>
EIK_HD void expand_box(G& g)
{
    int moved;
    do {
        moved = 0;
        if (g.Y0 > 0) { g.Y0--; g.note(sweep_line<1>(g.view(), g.my, g.Y0, -1, 0, g.X1, g.cnt)); moved++; }
        if (g.X1 < g.mx) { g.X1++; g.note(sweep_line<0>(g.view(), g.mx, g.X1, 1, g.Y0, g.Y1, g.cnt)); moved++; }
        if (g.Y1 < g.my) { g.Y1++; g.note(sweep_line<1>(g.view(), g.my, g.Y1, 1, 0, g.X1, g.cnt)); moved++; }
    } while (moved);
}

// reference init_cellh, src/time_2d.c:791-802
EIK_HD float head_in_cell(float vh, float vv, float hsc, float hsn)
{
    const float hsd = sqrtf(fmaf(-hsn, hsn, hsc * hsc));
    if (vh * hsd > vv * hsn) return fmaf(vh, hsn, vv * hsd);
    return kInf;
}

// reference init_cell (src/time_2d.c:758-789) for a source that sits on a corner of the
// cell: (dx,dy) in {0,1}^2 is the offset from corner (x,y) to the source.
template <class G>
EIK_HD void seed_cell(const G& g, int dx, int dy, int x, int y)
{
    const float hs0 = g.S(x, y);
    const float fdx = (float)dx, fdy = (float)dy, odx = (float)(1 - dx), ody = (float)(1 - dy);
    float hs1, est;
    // corner distances are 0, 1 or sqrt(2) cell units
    const float dist[3] = {0.f, hs0, hs0 * kSqrt2};
    est = dist[dx + dy];             if (est < g.T(x, y)) g.T(x, y) = est;
    est = dist[(1 - dx) + dy];       if (est < g.T(x + 1, y)) g.T(x + 1, y) = est;
    est = dist[dx + (1 - dy)];       if (est < g.T(x, y + 1)) g.T(x, y + 1) = est;
    est = dist[(1 - dx) + (1 - dy)]; if (est < g.T(x + 1, y + 1)) g.T(x + 1, y + 1) = est;
    if (x && (hs1 = g.S(x - 1, y)) < hs0) {
        if ((est = head_in_cell(fdx, fdy, hs0, hs1)) < g.T(x, y)) g.T(x, y) = est;
        if ((est = head_in_cell(fdx, ody, hs0, hs1)) < g.T(x, y + 1)) g.T(x, y + 1) = est;
    }
    if (y && (hs1 = g.S(x, y - 1)) < hs0) {
        if ((est = head_in_cell(fdy, fdx, hs0, hs1)) < g.T(x, y)) g.T(x, y) = est;
        if ((est = head_in_cell(fdy, odx, hs0, hs1)) < g.T(x + 1, y)) g.T(x + 1, y) = est;
    }
    if (x < g.my - 1 && (hs1 = g.S(x + 1, y)) < hs0) {   // sic: the reference compares x with nmesh_y (:781)
        if ((est = head_in_cell(odx, fdy, hs0, hs1)) < g.T(x + 1, y)) g.T(x + 1, y) = est;
        if ((est = head_in_cell(odx, ody, hs0, hs1)) < g.T(x + 1, y + 1)) g.T(x + 1, y + 1) = est;
    }
    if (y < g.my - 1 && (hs1 = g.S(x, y + 1)) < hs0) {
        if ((est = head_in_cell(ody, fdx, hs0, hs1)) < g.T(x, y + 1)) g.T(x, y + 1) = est;
        if ((est = head_in_cell(ody, odx, hs0, hs1)) < g.T(x + 1, y + 1)) g.T(x + 1, y + 1) = est;
    }
}

// Geometry of the half-spacing grid along one axis (src/time_2d.c:844-864).
EIK_HD void refine_axis(int s_coarse, int n_coarse, int* n, int* src, int* c0, int* half)
{
    int d;
    *n = kFineMax;
    *src = 2 * kInitMin + 1;
    *half = 1;
    *c0 = s_coarse - kInitMin - 1;
    if ((d = kInitMin - s_coarse) >= 0) {
        *c0 += d + 1;
        d = 1 + 2 * d;
        *n -= d;
        *src -= d;
        *half = 0;
    }
    if ((d = s_coarse + kInitMin - n_coarse + 1) >= 0) *n -= 1 + 2 * d;
}

// Initialisation round the source (reference init_point, src/time_2d.c:503-717), in two steps.
// seed_search: the largest quasi-homogeneous box round the source and what to do with it.
enum SeedKind : int { kSeedBox = 0, kSeedNearest = 1, kSeedRefine = 2 };

template <class G>
EIK_HD int seed_search(G& g, bool allow_refine)
{
    const int mx = g.mx, my = g.my, ys = g.ys;
    const int ysc = (ys == my) ? ys - 1 : ys;
    const float hs0 = g.S(0, ysc);
    const float tol = hs0 * 0.001f;   // eps_init of src/misfit.c:278
    int failN = 0, failS = 0, tried;
    int X1 = 0, Y0 = ysc, Y1 = ysc;
    // In a depth-only medium a new column can never fail and a new row is one test (:598-644).
    do {
        tried = 0;
        if (Y0 && !failN) {
            tried++;
            --Y0;
            if (fabsf(g.S(0, Y0) - hs0) > tol) { failN = 1; Y0++; }
        }
        if (X1 < mx - 1) { tried++; ++X1; }
        if (Y1 < my - 1 && !failS) {
            tried++;
            ++Y1;
            if (fabsf(g.S(0, Y1) - hs0) > tol) { failS = 1; Y1--; }
        }
        if (tried && (failN + failS)) tried = 0;
    } while (tried);
    X1++;
    Y1++;
    if (failN) Y0++;
    if (failS) Y1--;
    if (Y0 > ys || Y1 < ys) { Y0 = ysc; X1 = 1; Y1 = ysc + 1; }   // X1 >= 1 > xs = 0 always
    g.X1 = X1; g.Y0 = Y0; g.Y1 = Y1;
    if (!allow_refine ||
        ((Y0 == 0 || (ys - Y0) >= kInitMin) && (X1 == mx || X1 >= kInitMin) && (Y1 == my || (Y1 - ys) >= kInitMin)))
        return (X1 * (Y1 - Y0) == 1) ? kSeedNearest : kSeedBox;
    return kSeedRefine;
}

// exact time of node (x,y) in the homogeneous box round the source (src/time_2d.c:695-699)
EIK_HD float box_time(float hs0, int x, int dy)
{
    const float fy = (float)dy;
    const float sq = fmaf((float)x, (float)x, fy * fy);   // exact: small integers
    const float s = sqrtf(sq);
#ifdef EIK_COMPENSATED
    if (s > 0.f) {
        const float c = fmaf(-s, s, sq) * (0.5f / s);
        return fmaf(hs0, s, hs0 * c);
    }
#endif
    return hs0 * s;
}

template <class G>
EIK_HD float source_slowness(const G& g) { return g.S(0, (g.ys == g.my) ? g.ys - 1 : g.ys); }

// seed_fill: times of the box found by seed_search (kinds kSeedBox and kSeedNearest).
template <class G>
EIK_HD void seed_fill(G& g, int kind)
{
    const int ys = g.ys;
    if (kind == kSeedNearest) {
        // reference init_nearest for a node source on the left edge (:733-739)
        EIK_CNT(g, nearest_init);
        if (0 < g.mx && ys < g.my) seed_cell(g, 0, 0, 0, ys);
        if (0 < g.mx && ys) seed_cell(g, 0, 1, 0, ys - 1);
    } else {
        EIK_CNT(g, box_init);
        const float hs0 = source_slowness(g);
        for (int x = 0; x <= g.X1; x++)
            for (int y = g.Y0; y <= g.Y1; y++) g.T(x, y) = box_time(hs0, x, y - ys);
    }
}

// Returns true when the re-discretised initialisation is required.
template <class G>
EIK_HD bool seed_source(G& g, bool allow_refine)
{
    const int kind = seed_search(g, allow_refine);
    if (kind == kSeedRefine) return true;
    seed_fill(g, kind);
    return false;
}

// Complete solve of one source.  `t` must hold nx*ny nodes, `tf` (kFineMax*22 nodes is
// enough: the refined grid of a left-edge source has 22 columns at most) the refined grid.
EIK_HD int solve(const float* s, int sstride, int nx, int ny, int iz, float* t, float* tf, int ts, Counters* cnt)
{
    if (nx < 2 || ny < 2) return kErrDim;
    Grid<CoarseMedium> g;
    g.t = t; g.ts = ts; g.nx = nx; g.ny = ny; g.mx = nx - 1; g.my = ny - 1;
    g.S = CoarseMedium{s, sstride, nx - 1, ny - 1};
    g.ys = iz; g.status = kOk; g.cnt = cnt;
    for (int i = 0; i < nx * ny; i++) t[(size_t)i * ts] = kInf;

    if (seed_source(g, true)) {
        // reference recursive_init, src/time_2d.c:806-917
        EIK_CNT(g, recursive_init);
        int nxf, nyf, xsf, ysf, i0, j0, hx, hy;
        refine_axis(0, nx, &nxf, &xsf, &i0, &hx);
        refine_axis(iz, ny, &nyf, &ysf, &j0, &hy);
        if (nxf < 2 || nyf < 2) return kErrRecurs;
        Grid<FineMedium> f;
        f.t = tf; f.ts = ts; f.nx = nxf; f.ny = nyf; f.mx = nxf - 1; f.my = nyf - 1;
        f.S = FineMedium{g.S, j0, hy};
        f.ys = ysf; f.status = kOk; f.cnt = cnt;
        for (int i = 0; i < nxf * nyf; i++) tf[(size_t)i * ts] = kInf;
        seed_source(f, false);
        expand_box(f);
        if (f.status != kOk) g.status = f.status;
        for (int i = 0, ii = 0; ii < nxf; ii += 2, i++)
            for (int j = j0 + hy, jj = hy; jj < nyf; jj += 2, j++) g.T(i, j) = f.T(ii, jj);
        g.X1 = (kInitMin < g.mx) ? kInitMin : g.mx;
        g.Y0 = (iz - kInitMin > 0) ? iz - kInitMin : 0;
        g.Y1 = (iz + kInitMin < g.my) ? iz + kInitMin : g.my;
    }
    expand_box(g);
    return g.status;
}

}  // namespace eik
