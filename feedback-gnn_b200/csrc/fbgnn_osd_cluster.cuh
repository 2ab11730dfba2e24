// fbgnn_osd_cluster.cuh -- OSD for bases whose reduced matrix [H_perm | s] exceeds the shared memory of one SM.
//
// A thread-block cluster of C CTAs (2, 4 or 8 SMs) decodes ONE frame and computes exactly what k_osd computes, for
// every order (GF(2) elimination and integer weights: the outputs are bit-identical).
//   - Every CTA runs k_osd's sort on its own, so every CTA holds order / inv without an exchange.
//   - The R basis rows are cut into C contiguous ranges of rs rows, rs a multiple of 32 so that no 32-row bit-vector
//     word of the OSD-CS sweep straddles two CTAs.  CTA q builds and keeps rows [q rs, (q + 1) rs) of the matrix,
//     word-major with an odd row stride as k_osd does.  On small bases the last CTAs own no rows; they still pass
//     every barrier.
//   - Elimination, one cluster barrier per basis row r: the owner of row r (the only CTA that ever wrote it) finds the
//     pivot and copies it and the row into slot r & 1 of its shared memory; after the barrier every CTA copies the
//     slot through distributed shared memory (DSMEM), records the pivot and XORs the row into its own rows.  Slot
//     r & 1 is written next at step r + 2, by a CTA that has passed barrier r + 1, which every CTA reaches only after
//     it has finished reading the slot at step r.
//   - OSD-CS: every CTA knows all pivots and lists the non-pivot columns itself.  It adds its rows' share of each
//     single-column weight into rank 0's csum with DSMEM atomics (integer sums: order-independent) and stores its
//     32-row words of s' and of the first lp non-pivot columns into rank 0's sv / cv.  Rank 0 scores the OSD-0 and
//     single candidates from these and the pairs with k_osd's own code (osd_cs_best); the other CTAs read the winner
//     from rank 0 after one more barrier.
//   - Output: the frame's outputs are cleared (each CTA a slice of the variables), one barrier, then each CTA writes
//     the solution of its own pivot rows and rank 0 the winner's columns t0 / t1.
// No CTA returns early: every CTA executes every cluster barrier.
#pragma once
#include <cooperative_groups.h>

#include "fbgnn_kernels.cuh"

namespace fbgnn {

constexpr int OSD_CL_MAX = 8;           // largest portable cluster

struct OsdCluster {
    int C;                              // CTAs per frame
    int rs;                             // basis rows per CTA, a multiple of 32
    int slot_off;                       // byte offset of the broadcast slots in dynamic shared memory
};

// Dynamic shared memory of every CTA (rs_p = rs | 1, W = ceil((n + 1) / 32)):
//   max(npad * 8, W * rs_p * 4) bytes shared by the sort keys and this CTA's rows of the matrix; u16 order[n], inv[n],
//   piv[R]; at slot_off u32 slot[2][W + 1] (words of the broadcast row, then its pivot), row[W + 1] (this CTA's copy of
//   the current pivot row), svl[rs / 32] (s' over this CTA's rows); with order > 0, at cv_off (used on rank 0 only)
//   u32 cv[lp][RW], sv[RW] and int csum[n] (the single-column weights, less one).
static __global__ void __launch_bounds__(256, 1) k_osd_cluster(const OsdArgs a, const OsdCluster P) {
    extern __shared__ unsigned long long osd_smem[];
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int n = a.S.n, R = a.S.m, T = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = T >> 5;
    const int C = P.C, rank = (int)cluster.block_rank(), RS = P.rs;
    const int W = (n + 1 + 31) / 32, Rp = RS | 1;                // odd stride: no bank conflicts across words
    const int r0 = min(rank * RS, R), nr = min(R - r0, RS);      // this CTA's basis rows [r0, r0 + nr)
    const int64_t fi = blockIdx.x / C;
    const int64_t b = a.frame_list ? a.frame_list[fi] : fi;
    unsigned long long *keys = osd_smem;
    uint32_t *M = (uint32_t *)osd_smem;
    const size_t main_bytes = ((size_t)a.npad * 8 > (size_t)W * Rp * 4) ? (size_t)a.npad * 8 : (size_t)W * Rp * 4;
    uint16_t *order = (uint16_t *)((uint8_t *)osd_smem + ((main_bytes + 7) & ~(size_t)7));
    uint16_t *inv = order + n, *piv = inv + n;
    uint32_t *slot = (uint32_t *)((uint8_t *)osd_smem + P.slot_off), *row = slot + 2 * (W + 1), *svl = row + (W + 1);
    const int RW = (R + 31) / 32, lp = min(a.order, max(n - R, 0));
    uint32_t *cv = (uint32_t *)((uint8_t *)osd_smem + a.cv_off), *sv = cv + (size_t)lp * RW;    // rank 0's OSD-CS vectors
    int *csum = (int *)(sv + RW);                                                                // and single weights

    // 1. + 2. the sort, and this CTA's rows of the permuted [H | s]
    osd_sort(a, b, keys, order, inv);
    osd_build_rows(a, b, M, Rp, inv, r0, nr);
    if (a.order > 0 && rank == 0)
        for (int i = tid; i < n; i += T) csum[i] = 0;
    cluster.sync();                                              // every CTA runs before any DSMEM access; csum is clear

    // 3. row-wise elimination, one cluster barrier per basis row
    const int wn = n >> 5;
    const uint32_t last_mask = (n & 31) ? ((1u << (n & 31)) - 1u) : 0u;   // columns < n inside word wn
    for (int r = 0; r < R; r++) {
        const int owner = r / RS;
        uint32_t *sl = slot + (r & 1) * (W + 1);
        if (rank == owner && tid < 32) {
            const int lr = r - r0;
            const int p = osd_pivot(M, Rp, lr, W, wn, last_mask, tid);
            for (int w = (p >> 5) + tid; w < W; w += 32) sl[w] = M[w * Rp + lr];   // the row is zero before word p / 32
            if (tid == 0) sl[W] = (uint32_t)p;
        }
        cluster.sync();
        const uint32_t *src = cluster.map_shared_rank(sl, owner);
        for (int w = tid; w <= W; w += T) row[w] = src[w];
        __syncthreads();
        const int p = (int)row[W], pw = p >> 5;
        const uint32_t pm = 1u << (p & 31);
        if (tid == 0) piv[r] = (uint16_t)p;
        for (int i = tid; i < nr; i += T) {
            if (r0 + i != r && (M[pw * Rp + i] & pm)) {
                for (int w = pw; w < W; w++) M[w * Rp + i] ^= row[w];
            }
        }
        __syncthreads();
    }

    // 4. OSD-CS: the candidate of least (weight, index); t0 / t1 are its columns (-1: none)
    int t0 = -1, t1 = -1;
    if (a.order > 0) {
        __shared__ unsigned long long best;
        __shared__ int num_np;
        uint32_t *cv0 = cluster.map_shared_rank(cv, 0), *sv0 = cluster.map_shared_rank(sv, 0);
        int *csum0 = cluster.map_shared_rank(csum, 0);
        const int NK = (nr + 31) / 32, k0 = r0 / 32;             // this CTA's 32-row words: k0 .. k0 + NK - 1
        // 4a. the non-pivot columns listed in inv (free since step 2); s' over this CTA's rows, here and on rank 0
        if (tid == 0) best = ~0ull;
        osd_cs_list(inv, piv, n, R, &num_np);
        for (int k = warp; k < NK; k += nw) {
            const int i = k * 32 + lane;
            const uint32_t v = __ballot_sync(0xffffffffu, i < nr && ((M[wn * Rp + i] >> (n & 31)) & 1u));
            if (lane == 0) { svl[k] = v; sv0[k0 + k] = v; }
        }
        __syncthreads();
        const int N = num_np;
        // 4b. single columns: this CTA's rows' share of each weight, and its words of the first lp columns, to rank 0
        for (int i = warp; i < N; i += nw) {
            const int c = inv[i], cw = c >> 5;
            const uint32_t cm = 1u << (c & 31);
            int w = 0;
            for (int k = 0; k < NK; k++) {
                const int j = k * 32 + lane;
                const uint32_t v = __ballot_sync(0xffffffffu, j < nr && (M[cw * Rp + j] & cm));
                if (i < lp && lane == 0) cv0[i * RW + k0 + k] = v;
                w += __popc(v ^ svl[k]);
            }
            if (lane == 0 && w) atomicAdd(&csum0[i], w);
        }
        cluster.sync();
        // 4c. rank 0: OSD-0, the singles and (k_osd's code) the pairs
        if (rank == 0) {
            unsigned long long mine = ~0ull;
            if (tid == 0) {                                      // the empty set: OSD-0
                int w = 0;
                for (int k = 0; k < RW; k++) w += __popc(sv[k]);
                mine = (unsigned long long)w << 32;
            }
            for (int i = tid; i < N; i += T) mine = min(mine, ((unsigned long long)(1 + csum[i]) << 32) | (uint32_t)(1 + i));
            osd_cs_best(mine, cv, sv, RW, lp, N, &best);
        }
        cluster.sync();
        osd_cs_columns((uint32_t)*cluster.map_shared_rank(&best, 0), N, lp, inv, t0, t1);
    }

    // 5. clear the frame's outputs (a slice of the variables per CTA), then the solution of this CTA's pivot rows; rank
    //    0 adds t0 / t1.  The barrier orders the clears before every CTA's stores, and it is the last one: no CTA reads
    //    another's shared memory after it, so a CTA may exit once past it.
    const int v0 = (int)((int64_t)n * rank / C), v1 = (int)((int64_t)n * (rank + 1) / C);
    if (a.e_hat.ptr) for (int v = v0 + tid; v < v1; v += T) a.e_hat(b, v) = 0;
    if (a.vbits) for (int v = v0 + tid; v < v1; v += T) a.vbits[b * n + v] &= (uint8_t)~(1u << a.vbit);
    cluster.sync();
    osd_write_solution(a, b, M, Rp, order, piv + r0, nr, t0, t1, rank == 0);
}

}  // namespace fbgnn
