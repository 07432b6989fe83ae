// eik_march.cuh -- the column march of the eikonal solver with its columns in TENSOR MEMORY (sm_100a, device only).
//
// After the expanding box spans the whole depth range a solve is a march over columns: column x+1 from column x and the
// slowness column (eik_fast.cuh: march_sweep3).  Its accesses are warp-uniform in the index -- every lane is at the same
// depth at the same time -- which is exactly the 32x32b shape of tcgen05.ld / tcgen05.st: thread i of a warp reads or
// writes 32 bits of TMEM lane (32*(warp%4) + i) at a column address common to the warp.  So the past column, the current
// column and the slowness column of a marching warp live in tensor memory, node k of a lane at column k+1 of that lane:
//   * a marching warp needs no shared memory, which goes to the warps that are in their box phase (per-lane indices):
//     eik_pipe_kernel (eikonal.cu) runs 12 warps per SM on 7 - 9 shared-memory slices + 8 TMEM sets instead of 9 warps
//     on the Example plane;
//   * four consecutive nodes move per instruction (.x4);
//   * TMEM load latency is 12 cycles against 29 for shared memory.
// A column array holds the nodes -1 .. CA-2 (CA = 64 for nz <= 62, CA = 128 for 88 <= nz <= 126; eikonal.cu: pipe_shape):
// nodes -1 and ke+1.. carry sentinels larger than any
// time (strictly increasing, so they never tie), which end the chains exactly where march_sweep3's kEdge slots do.
// Arithmetic: chain_a_node / chain_b_node of eik_fast.cuh, unchanged -- results are bit-identical to the fused kernel's.
#pragma once
#include <stdint.h>

#include "eik_fast.cuh"
#include "eikonal.cuh"

namespace eikm {

using eikf::kEdge;
using eikf::kInf;

// The column count is an immediate: the toolchain derives the kernel's tensor-memory footprint (and with it the
// number of co-resident CTAs) from it.
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst)   // whole warp, one warp per CTA
{
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "n"(NCOLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&v)[4])
{
    uint32_t r0, r1, r2, r3;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(taddr));
    v[0] = __uint_as_float(r0); v[1] = __uint_as_float(r1); v[2] = __uint_as_float(r2); v[3] = __uint_as_float(r3);
}
__device__ __forceinline__ float tmem_ld1(uint32_t taddr)
{
    uint32_t r0;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r0) : "r"(taddr));
    return __uint_as_float(r0);
}
// The registers of a tcgen05.ld are valid after the wait; tying them to it keeps their uses behind it.
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld(float (&a)[4])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(a[0]), "+f"(a[1]), "+f"(a[2]), "+f"(a[3])::"memory");
}
__device__ __forceinline__ void tmem_wait_ld(float (&a)[4], float (&b)[4])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(a[0]), "+f"(a[1]), "+f"(a[2]), "+f"(a[3]), "+f"(b[0]), "+f"(b[1]), "+f"(b[2]), "+f"(b[3])::"memory");
}
__device__ __forceinline__ void tmem_wait_ld(float (&a)[4][4])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+f"(a[0][0]), "+f"(a[0][1]), "+f"(a[0][2]), "+f"(a[0][3]), "+f"(a[1][0]), "+f"(a[1][1]), "+f"(a[1][2]), "+f"(a[1][3]),
                   "+f"(a[2][0]), "+f"(a[2][1]), "+f"(a[2][2]), "+f"(a[2][3]), "+f"(a[3][0]), "+f"(a[3][1]), "+f"(a[3][2]), "+f"(a[3][3])::"memory");
}
__device__ __forceinline__ void tmem_wait_ld(float& a) { asm volatile("tcgen05.wait::ld.sync.aligned;" : "+f"(a)::"memory"); }
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const float (&v)[4])
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(__float_as_uint(v[0])),
                 "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3]))
                 : "memory");
}
__device__ __forceinline__ void tmem_st1(uint32_t taddr, float v)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(__float_as_uint(v)) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// value of a sentinel node (k < 0 or k > ke): above every travel time, strictly increasing with k
__device__ __forceinline__ float sentinel(int k, int ke) { return k < 0 ? kEdge : kEdge * (1.0f + (float)(k - ke) * (1.0f / 1024.0f)); }

// One group of four nodes of each chain (see tmem_sweep).  SECOND: the other chain has been at these nodes, its values
// are read back and merged; in the first half of a column there is nothing to merge (a real node's value never exceeds
// INF, so the merge with INF it would be is the identity).
struct SweepRegs {
    float pa_cur[4], pb_cur[4], sa_cur[4], sb_cur[4];
};

template <int NB, bool MASKED, bool SECOND>
__device__ __forceinline__ void tmem_group(int j, bool need, uint32_t tp, uint32_t tc, uint32_t tS, eikf::ChainA& a, eikf::ChainB& b,
                                           SweepRegs& r, bool& tie)
{
    float pa_nxt[4], pb_nxt[4], ca_old[4], cb_old[4], sa_nxt[4], sb_nxt[4];
    if (j + 1 < NB) {
        tmem_ld4(tp + 4 * (j + 1), pa_nxt); tmem_ld4(tp + 4 * (NB - 2 - j), pb_nxt);
        tmem_ld4(tS + 4 * (j + 1), sa_nxt); tmem_ld4(tS + 4 * (NB - 2 - j), sb_nxt);
    } else {
#pragma unroll
        for (int c = 0; c < 4; c++) { pa_nxt[c] = 4.0f * kEdge; pb_nxt[c] = 2.0f * kEdge; sa_nxt[c] = kInf; sb_nxt[c] = kInf; }
    }
    if (SECOND) { tmem_ld4(tc + 4 * j, ca_old); tmem_ld4(tc + 4 * (NB - 1 - j), cb_old); }
    tmem_wait_ld(pa_nxt, pb_nxt);
    if (SECOND) tmem_wait_ld(ca_old, cb_old);
    tmem_wait_ld(sa_nxt, sb_nxt);
    float va[4], vb[4];
#pragma unroll
    for (int c = 0; c < 4; c++) {
        // chain A at node 4j-1+c: its cell is column 4j+c of the slowness array = element c of group j
        const float own_a = a.pk;
        float v = eikf::chain_a_node(a, (c < 3) ? r.pa_cur[c + 1] : pa_nxt[0], r.sa_cur[c], tie);
        if (SECOND) v = fminf(v, ca_old[c]);
        va[c] = (MASKED && !need) ? own_a : v;
        // chain B at node kb = CA-2-4j-c: cell kb-1 is column kb of the slowness array = element 2-c of group NB-1-j
        // (c < 3), element 3 of the next lower group (c == 3)
        const float own_b = b.pk;
        float w = eikf::chain_b_node(b, (c < 3) ? r.pb_cur[2 - c] : pb_nxt[3], (c < 3) ? r.sb_cur[2 - c] : sb_nxt[3]);
        if (SECOND) w = fminf(w, cb_old[3 - c]);
        vb[3 - c] = (MASKED && !need) ? own_b : w;
    }
    tmem_st4(tc + 4 * j, va);
    tmem_st4(tc + 4 * (NB - 1 - j), vb);
#pragma unroll
    for (int c = 0; c < 4; c++) { r.pa_cur[c] = pa_nxt[c]; r.pb_cur[c] = pb_nxt[c]; r.sa_cur[c] = sa_nxt[c]; r.sb_cur[c] = sb_nxt[c]; }
}

// One column: past column in TMEM array tp, new column into array tc, slowness cells in array tS (cell k at column k+1,
// cells -1 and ke.. = INF); all three are column addresses of this warp's lane quarter.
// MASKED: lanes with need == false keep their past column (their box phase ended at a later column than the others').
template <int NB, bool MASKED>
__device__ __forceinline__ bool tmem_sweep(bool need, uint32_t tp, uint32_t tc, uint32_t tS)
{
    bool tie = false;
    SweepRegs r;
    tmem_ld4(tp, r.pa_cur);
    tmem_ld4(tp + 4 * (NB - 1), r.pb_cur);
    tmem_ld4(tS, r.sa_cur);
    tmem_ld4(tS + 4 * (NB - 1), r.sb_cur);
    tmem_wait_ld(r.pa_cur, r.pb_cur);
    tmem_wait_ld(r.sa_cur, r.sb_cur);
    // chain A starts at node -1 (parent -2: nothing there), chain B at node CA-2 (parent CA-1: nothing there)
    eikf::ChainA a{2.0f * kEdge, r.pa_cur[0], kInf, kInf};
    eikf::ChainB b{4.0f * kEdge, r.pb_cur[3], kInf, kInf};
    // (unrolling these loops by two saves the register copies between the group being worked on and the one being fetched,
    //  7 % of the instructions, and measured 2 - 8 % SLOWER: profiles/README.md, r2unroll)
#pragma unroll 1
    for (int j = 0; j < NB / 2; j++) tmem_group<NB, MASKED, false>(j, need, tp, tc, tS, a, b, r, tie);
    tmem_wait_st();                      // the other chain's stores must have landed before they are read back
#pragma unroll 1
    for (int j = NB / 2; j < NB; j++) tmem_group<NB, MASKED, true>(j, need, tp, tc, tS, a, b, r, tie);
    return need && tie;
}

}  // namespace eikm
