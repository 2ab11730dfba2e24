// fbgnn_gnn_tc.cuh -- tensor-core (tcgen05 / TMEM) form of the feedback GNN's dense products, sm_100a.
//
// Feedback_GNN.call (feedback_gnn.py:161-188) per variable node: six edge MLPs whose first layer is rank one in the
// check feature (thread-local FMAs + tanh), and then three dense products with the weights as the stationary operand:
//     [hidden sums of the x edges, 40] x W2x [40 x 20],  [.. of the z edges, 40] x W2z [40 x 20],
//     [m_x, m_z, 40] x W3[0:40] [40 x 40]                       (the three prior features of W3 stay thread-local).
// Rows = frames x variable nodes: the one place on the headline path where "frames x nodes x hidden" is a real dense
// GEMM (north star; SURVEY.md A8).  Same machinery as GNN_BP4's tensor-core path (fbgnn_gbp_tc.cuh): a group of 128
// threads owns 128 rows, thread r <-> row r <-> TMEM lane r; the A operand goes registers -> TMEM (tcgen05.st), the
// weights sit in shared memory as TF32 hi / lo tiles in the canonical K-major UMMA layout (staged by one bulk-async
// copy), D accumulates in TMEM; float32 accuracy from TF32 hardware by the three-product split.
//
// Selected by Feedback_GNN(..., gemm="tf32x3") / fbgnn_gnn_set_gemm (what bench.py runs).  The arithmetic of a
// tcgen05.mma kind::tf32 step is an integer model characterised on B200 (csrc/fb_umma.h), so the CPU oracle reproduces
// this kernel BIT FOR BIT (oracle/fbgnn_oracle.c gnn_frame_tc mirrors it operation by operation); against the FMA kernel
// k_gnn the outputs agree to float32 re-association accuracy (5e-7).  tests/test_gpu_gnn_tc.py.
#ifndef FBGNN_GNN_TC_CUH
#define FBGNN_GNN_TC_CUH

#include "fbgnn_gbp_tc.cuh"

namespace fbgnn {
namespace tc {

struct GnnW {                                  // offsets in floats; each operand: [hi tile][lo tile]
    static constexpr int H = 40, M = 20;
    static constexpr int W2X = 0, W2Z = W2X + t(40, 32);              // K = H, N = M (32)
    static constexpr int W3AB = W2Z + t(40, 32);                      // K = 2M, N = H (48)
    static constexpr int SCALAR = W3AB + t(40, 48);                   // GnnLayout<40, 20> block (first layers, biases, W3 rows 40..42, W0)
    static constexpr int total = SCALAR + GnnLayout<40, 20>::total;
};

// One side's edge phase of a tile row: hidden sums over the DV edges, 8 hidden units at a time, straight into TMEM as
// the A operand of the W2 product (hi at [0, 40), lo at [40, 80)).  The first-layer rows of units j, j+1 (j even) sit
// interleaved in this blob, {w_cn, w_Lx, w_Ly, w_Lz} of j in the even and of j+1 in the odd positions (fbgnn_gnn.cu), so
// that in paired arithmetic (MATH::kPaired) the two units go through the same float2 instructions with no moves.
template <int DV, typename MATH>
__device__ __forceinline__ void gnn_edges_tc(const Grp &g, const float *__restrict__ w1p, const float *__restrict__ b1,
                                             const float hc[DV], float f1, float f2, float f3) {
    constexpr int H = 40, JB = 8;
#pragma unroll 1
    for (int j0 = 0; j0 < H; j0 += JB) {
        uint32_t hi[JB], lo[JB];
#pragma unroll
        for (int q = 0; q < JB; q += 2) {
            const float4 wa = *reinterpret_cast<const float4 *>(w1p + 4 * (j0 + q));       // {cn_j, cn_j+1, Lx_j, Lx_j+1}
            const float4 wb = *reinterpret_cast<const float4 *>(w1p + 4 * (j0 + q) + 4);   // {Ly_j, Ly_j+1, Lz_j, Lz_j+1}
            float2 hs;
            if constexpr (MATH::kPaired) {
                const float2 wcn = make_float2(wa.x, wa.y);
                const float2 base = FB_FMA2(fb2s(f3), make_float2(wb.z, wb.w), FB_FMA2(fb2s(f2), make_float2(wb.x, wb.y),
                                            FB_FMA2(fb2s(f1), make_float2(wa.z, wa.w), make_float2(b1[j0 + q], b1[j0 + q + 1]))));
                hs = MATH::tanh2(FB_FMA2(fb2s(hc[0]), wcn, base));
#pragma unroll
                for (int k = 1; k < DV; k++) hs = FB_ADD2(hs, MATH::tanh2(FB_FMA2(fb2s(hc[k]), wcn, base)));
            } else {
                const float base0 = FB_FMA(f3, wb.z, FB_FMA(f2, wb.x, FB_FMA(f1, wa.z, b1[j0 + q])));     // bias first
                const float base1 = FB_FMA(f3, wb.w, FB_FMA(f2, wb.y, FB_FMA(f1, wa.w, b1[j0 + q + 1])));
                hs.x = MATH::tanh(FB_FMA(hc[0], wa.x, base0));
                hs.y = MATH::tanh(FB_FMA(hc[0], wa.y, base1));
#pragma unroll
                for (int k = 1; k < DV; k++) {
                    hs.x = FB_ADD(hs.x, MATH::tanh(FB_FMA(hc[k], wa.x, base0)));
                    hs.y = FB_ADD(hs.y, MATH::tanh(FB_FMA(hc[k], wa.y, base1)));
                }
            }
            const float2 h = make_float2(tf32_hi(hs.x), tf32_hi(hs.y));
            const float2 l = MATH::kPaired ? FB_SUB2(hs, h) : make_float2(FB_SUB(hs.x, h.x), FB_SUB(hs.y, h.y));
            hi[q] = __float_as_uint(h.x); hi[q + 1] = __float_as_uint(h.y);
            lo[q] = __float_as_uint(l.x); lo[q + 1] = __float_as_uint(l.y);
        }
        __syncwarp();
        tmem_st8(g.lane_base + j0, hi);
        tmem_st8(g.lane_base + H + j0, lo);
    }
}

// TMEM columns of a group: A operands at [0, 80) (hi, lo), D at [80, 128).
template <int DV, typename MATH>
__global__ void __launch_bounds__(256, 2) k_gnn_tc(const GnnArgs a, const float *__restrict__ wtc) {
    constexpr int H = 40, M = 20;
    typedef GnnLayout<H, M> Lay;
    extern __shared__ __align__(128) float sm[];
    __shared__ uint64_t bars[2];
    __shared__ uint32_t tslot;
    Grp g = cta_setup(sm, wtc, GnnW::total, bars, &tslot);
    const uint32_t sbase = smem_u32(sm);
    const float *ws = sm + GnnW::SCALAR;                        // scalar-path weights, GnnLayout offsets
    const int n = a.X.n, t = threadIdx.x & 127;
    const int64_t total = a.num_frames * n, ntiles = (total + 127) / 128;
    const float dg = (float)DV;
    // inputs of a row: the three prior features and the signed logits of its 2 DV checks; the next tile's are fetched
    // while the current tile is processed (the gathers are L2 latency)
    auto fetch = [&](int64_t tile, float &q1, float &q2, float &q3, float (&qx)[DV], float (&qz)[DV], int64_t &qb, int &qv) -> bool {
        const int64_t it = tile * 128 + t;
        const bool ok = tile < ntiles && it < total;
        q1 = q2 = q3 = 0.0f;
#pragma unroll
        for (int k = 0; k < DV; k++) { qx[k] = 0.0f; qz[k] = 0.0f; }
        qb = 0; qv = 0;
        if (ok) {
            const int64_t fi = it / n;
            qv = (int)(it - fi * n);
            qb = a.frame_list ? a.frame_list[fi] : fi;
            q1 = a.h_vn(qb, qv, 0); q2 = a.h_vn(qb, qv, 1); q3 = a.h_vn(qb, qv, 2);
#pragma unroll
            for (int k = 0; k < DV; k++) {
                const int cx = a.X.vn_cn[qv * DV + k], cz = a.Z.vn_cn[qv * DV + k];
                const float lx = a.logit_hx(cx, qb), lz = a.logit_hz(cz, qb);
                qx[k] = a.sx(cx, qb) ? -lx : lx;
                qz[k] = a.sz(cz, qb) ? -lz : lz;
            }
        }
        return ok;
    };
    float n1, n2, n3, nhx[DV], nhz[DV];
    int64_t nb;
    int nv;
    bool nvalid = fetch((int64_t)blockIdx.x * 2 + g.gid, n1, n2, n3, nhx, nhz, nb, nv);
    for (int64_t tile = (int64_t)blockIdx.x * 2 + g.gid; tile < ntiles; tile += (int64_t)gridDim.x * 2) {
        const bool valid = nvalid;
        const int64_t b = nb;
        const int v = nv;
        const float f1 = n1, f2 = n2, f3 = n3;
        float hcx[DV], hcz[DV];
#pragma unroll
        for (int k = 0; k < DV; k++) { hcx[k] = nhx[k]; hcz[k] = nhz[k]; }
        nvalid = fetch(tile + (int64_t)gridDim.x * 2, n1, n2, n3, nhx, nhz, nb, nv);
        float mm[2 * M];
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
            gnn_edges_tc<DV, MATH>(g, ws + (side ? Lay::W1tz : Lay::W1tx), ws + (side ? Lay::b1z : Lay::b1x),
                                   side ? hcz : hcx, f1, f2, f3);
            gemm(g, 0, H, H, 80, sbase + 4 * (side ? GnnW::W2Z : GnnW::W2X), 32, false);
            const float *b2 = ws + (side ? Lay::b2z : Lay::b2x);
#pragma unroll
            for (int c0 = 0; c0 < 24; c0 += 8) {
                float d[8];
                tmem_ld8(g.lane_base + 80 + c0, d);
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    if (c0 + q < M) {
                        // mean: the 1 / DV is folded into the W2 tiles (fbgnn_gnn.cu), so D already is the mean
                        const float r = (a.reduce == 0) ? FB_ADD(d[q], b2[c0 + q]) : FB_FMA(dg, b2[c0 + q], d[q]);
                        if (side == 0) mm[c0 + q] = r;
                        else mm[M + c0 + q] = r;
                    }
                }
            }
        }
        store_a<2 * M>(g, 0, 2 * M, mm);
        gemm(g, 0, 2 * M, 2 * M, 80, sbase + 4 * GnnW::W3AB, 48, false);
        float o0 = 0.0f, o1 = 0.0f, o2 = 0.0f;
#pragma unroll 1
        for (int c0 = 0; c0 < H; c0 += 8) {
            float d[8];
            tmem_ld8(g.lane_base + 80 + c0, d);
            if constexpr (MATH::kPaired) {          // units j, j+1 as one float2; o0 / o1 / o2 keep their j order
#pragma unroll
                for (int q = 0; q < 8; q += 2) {
                    const int j = c0 + q;
                    auto row = [&](int off) { return make_float2(ws[off + j], ws[off + j + 1]); };
                    float2 h = FB_FMA2(fb2s(f1), row(Lay::W3 + (2 * M) * H), make_float2(d[q], d[q + 1]));
                    h = FB_FMA2(fb2s(f2), row(Lay::W3 + (2 * M + 1) * H), h);
                    h = FB_FMA2(fb2s(f3), row(Lay::W3 + (2 * M + 2) * H), h);
                    h = MATH::tanh2(FB_ADD2(h, row(Lay::b3)));
                    o0 = FB_FMA(h.x, ws[Lay::W0 + j * 3 + 0], o0);
                    o1 = FB_FMA(h.x, ws[Lay::W0 + j * 3 + 1], o1);
                    o2 = FB_FMA(h.x, ws[Lay::W0 + j * 3 + 2], o2);
                    o0 = FB_FMA(h.y, ws[Lay::W0 + j * 3 + 3], o0);
                    o1 = FB_FMA(h.y, ws[Lay::W0 + j * 3 + 4], o1);
                    o2 = FB_FMA(h.y, ws[Lay::W0 + j * 3 + 5], o2);
                }
                continue;
            }
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const int j = c0 + q;
                float h = FB_FMA(f1, ws[Lay::W3 + (2 * M) * H + j], d[q]);
                h = FB_FMA(f2, ws[Lay::W3 + (2 * M + 1) * H + j], h);
                h = FB_FMA(f3, ws[Lay::W3 + (2 * M + 2) * H + j], h);
                h = MATH::tanh(FB_ADD(h, ws[Lay::b3 + j]));
                o0 = FB_FMA(h, ws[Lay::W0 + j * 3 + 0], o0);
                o1 = FB_FMA(h, ws[Lay::W0 + j * 3 + 1], o1);
                o2 = FB_FMA(h, ws[Lay::W0 + j * 3 + 2], o2);
            }
        }
        if (valid) {
            a.out(b, v, 0) = FB_ADD(o0, ws[Lay::b0 + 0]);
            a.out(b, v, 1) = FB_ADD(o1, ws[Lay::b0 + 1]);
            a.out(b, v, 2) = FB_ADD(o2, ws[Lay::b0 + 2]);
        }
    }
    cta_teardown(&tslot);
}

// Probe of ONE tcgen05.mma kind::tf32 step (M = 128, N = 16, K = 8): Dout = A B + Din for `trials` independent operand sets
// (A [T,128,8], B [T,8,16], Din / Dout [T,128,16]).  tests/test_gpu_gnn_tc.py compares what this GPU returns with the
// integer model of csrc/fb_umma.h.  One CTA of 128 threads.
static __global__ void __launch_bounds__(128) k_umma_probe(const float *A, const float *B, const float *Din, float *Dout,
                                                           int trials) {
    __shared__ __align__(128) float sb[128];
    __shared__ uint64_t bar;
    __shared__ uint32_t tslot;
    const int t = threadIdx.x, warp = t >> 5;
    if (warp == 0) tmem_alloc(&tslot, 32);
    if (t == 0) { mbar_init(&bar, 1); fence_async_smem(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = tslot, lane_base = tbase + ((uint32_t)(warp * 32) << 16);
    for (int tr = 0; tr < trials; tr++) {
        sb[b_tile_offset(t >> 3, t & 7, 8)] = B[(tr * 8 + (t & 7)) * 16 + (t >> 3)];
        uint32_t a[8], d0[8], d1[8];
#pragma unroll
        for (int q = 0; q < 8; q++) {
            a[q] = __float_as_uint(A[((int64_t)tr * 128 + t) * 8 + q]);
            d0[q] = __float_as_uint(Din[((int64_t)tr * 128 + t) * 16 + q]);
            d1[q] = __float_as_uint(Din[((int64_t)tr * 128 + t) * 16 + 8 + q]);
        }
        tmem_st8(lane_base + 0, a);
        tmem_st8(lane_base + 16, d0);
        tmem_st8(lane_base + 24, d1);
        tmem_wait_st();
        fence_async_smem();
        tc_fence_before();
        __syncthreads();
        if (t == 0) {
            tc_fence_after();
            umma_tf32_ts(tbase + 16, tbase + 0, b_desc(smem_u32(sb), 8), idesc_tf32(16), 1u);
            umma_commit(smem_u32(&bar));
        }
        mbar_wait(smem_u32(&bar), (uint32_t)(tr & 1));
        tc_fence_after();
        float v[8];
        tmem_ld8(lane_base + 16, v);
#pragma unroll
        for (int q = 0; q < 8; q++) Dout[((int64_t)tr * 128 + t) * 16 + q] = v[q];
        tmem_ld8(lane_base + 24, v);
#pragma unroll
        for (int q = 0; q < 8; q++) Dout[((int64_t)tr * 128 + t) * 16 + 8 + q] = v[q];
        tc_fence_before();
        __syncthreads();
    }
    if (warp == 0) tmem_dealloc(tbase, 32);
}

}  // namespace tc
}  // namespace fbgnn

#endif  // FBGNN_GNN_TC_CUH
