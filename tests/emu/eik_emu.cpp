// tests/emu/eik_emu.cpp -- TEST-ONLY host build of the CUDA solver core (csrc/eik_core.cuh).
// The very same source the GPU kernels instantiate is compiled for the CPU here, with
// contraction off, so that its FP32 results can be compared with the oracle at scale
// without a GPU.  Nothing in the product links this file.
#include "../../mcmc_eq_b200/csrc/eik_core.cuh"
#include <vector>
extern "C" int emu_time_2d(const float* s, int nx, int ny, int iz, float* t, int* counters)
{
    std::vector<float> tf(eik::kFineMax * 22);
    eik::Counters c = {};
    int rc = eik::solve(s, 1, nx, ny, iz, t, tf.data(), 1, counters ? &c : nullptr);
    if (counters) {
        counters[0] = c.col_sweeps; counters[1] = c.row_sweeps; counters[2] = c.reverse_sweeps;
        counters[3] = c.headwaves; counters[4] = c.recursive_init; counters[5] = c.nearest_init; counters[6] = c.box_init;
    }
    return rc;
}

// ---- host build of the warp-synchronous solver (csrc/eik_fast.cuh) with a 1-lane warp ----------------
#include "../../mcmc_eq_b200/csrc/eik_fast.cuh"
// gm != 0: the variant of the solver for slices in global memory (eik_fine_kernel): read-ahead row sweeps, columns of the
// growing box by the two-chain loop
// gm == 2: shared-memory slice with a second column buffer (Dims::lock_cols): lock-step columns without the read-ahead
static int g_gm = 0;
extern "C" void emu_set_gm(int on) { g_gm = on; }
extern "C" int emu_fast_time_2d(const float* s, int nx, int ny, int iz, float* t, const int* rows, int n_rows, float* rows_out)
{
    eikf::Dims D = eikf::make_dims(nx, ny);
    D.lock_cols = (g_gm == 2) ? 1 : 0;
    std::vector<float> SM(eikf::gmem_floats_per_lane(D)), W((size_t)D.wx * ny), WF(22 * 43);
    eikf::Lane L;
    if (g_gm == 1) eikf::carve_global(SM.data(), D, &L);
    else eikf::carve_shared(SM.data(), D, &L);
    L.W = W.data(); L.WF = WF.data();
    eikf::LaneTask task;
    task.valid = true; task.iz = iz; task.slow = s; task.out = rows_out; task.out_rstride = nx; task.full = t; task.hand_col = nullptr; task.hand_x1 = nullptr;
    return g_gm == 1 ? eikf::solve_warp<true, false>(D, L, task, rows, n_rows)
         : g_gm == 2 ? eikf::solve_warp<false, true>(D, L, task, rows, n_rows) : eikf::solve_warp<false, false>(D, L, task, rows, n_rows);
}
