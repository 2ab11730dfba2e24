// fbgnn_kernels.cuh -- sm_100a kernels of the BP -> feedback-GNN -> BP hot path.
//
// Layout in HBM (fused pipeline workspace, one row per frame):
//   vbits  u8  [B][n]        bit0 noise_x, bit1 noise_z, bit2 x_hat, bit3 z_hat
//   sbits  u8  [B][m_x+m_z]  syndrome_x then syndrome_z
//   L      f32 [B][3][n]     marginals (Lx, Ly, Lz) of the last BP stage
//   P      f32 [B][3][n]     priors produced by the feedback GNN for the next BP stage
//   logit  f32 [B][m_x+m_z]  z_logit (rows of hx) then x_logit (rows of hz)
//   active/rounds/flags u8 [B]
// Everything that is touched every BP iteration -- both message arrays, the per-variable
// priors, the syndrome bits -- lives in shared memory of the CTA that owns the frame; HBM is
// touched once per frame per stage.
//
// Arithmetic: float32, fixed evaluation order, all elementary functions from fb_math.h; the
// kernels are bit-exact against oracle/fbgnn_oracle.c (see tests/).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "fb_math.h"

namespace fbgnn {

typedef uint16_t idx_t;

// Tanner graph of one parity-check matrix, device pointers.
struct SideDev {
    int n, m, E;
    int reg_dv, reg_dc;        // common VN / CN degree if the side is regular, else 0
    const idx_t *vn_ptr;       // [n+1] edge ranges per VN; edges sorted by (vn, cn) = "VN order"
    const idx_t *vn_cn;        // [E]   check of each edge, VN order
    const idx_t *cn_ptr;       // [m+1] edge ranges per CN; edges sorted by (cn, vn) = "CN order"
    const idx_t *cn_edge;      // [E]   VN-order position of each edge, listed in CN order
    const idx_t *cn_vn;        // [E]   variable of each edge, listed in CN order
    const uint32_t *bitrows;   // [m][W] rows bit-packed, W = ceil(n/32)
    const int *h_vn_ptr;       // HOST copy of vn_ptr (launch-time partitioning of the cluster kernel; never read on the device)
};

template <typename T> struct View2 { T *ptr; int64_t s0, s1;
    __device__ __forceinline__ T &operator()(int64_t i, int64_t j) const { return ptr[i * s0 + j * s1]; } };
template <typename T> struct View3 { T *ptr; int64_t s0, s1, s2;
    __device__ __forceinline__ T &operator()(int64_t i, int64_t j, int64_t k) const { return ptr[i * s0 + j * s1 + k * s2]; } };

// ------------------------------------------------------------------ Philox4x32-10 ----
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ float u01(uint32_t r) { return (float)(r >> 8) * 5.9604644775390625e-08f; }

// ------------------------------------------------------------------ math policies -----
// MathExact: exp / log as polynomials on the FP32 pipe (fb_math.h, the restatement of Eigen's CPU kernels TF runs).
// MathSfu  : exp / log on the special-function unit (MUFU.EX2 / MUFU.LG2 with range reductions that confine the MUFU
//            inputs to finite sets; fb_math.h "SFU arithmetic").  2-3 ulp instead of 1, ~2.3x fewer instructions
//            per transcendental.
// Both are bit-identical to the CPU oracle in the same arithmetic (the oracle evaluates the MUFU through tables
// measured on the hardware), both carry the reference's saturation constants exactly, and the published logical
// error rates are reproduced in both (tests/test_gpu_sfu.py).
struct MathExact {
    static constexpr bool kSharedVnCorr = false;       // the reference's per-edge logaddexp
    static constexpr bool kPaired = false;             // FP32-pipe-bound: packed FP32 loses here (see WSmem)
    static __device__ __forceinline__ float softplus(float x) { return fb_softplusf(x); }
    static __device__ __forceinline__ float logaddexp(float a, float b) { return fb_logaddexpf(a, b); }
    static __device__ __forceinline__ float phi4(float x) { return fb_phi4f(x); }
    static __device__ __forceinline__ float phi2(float x) { return fb_phi2f(x); }
    static __device__ __forceinline__ float tanh(float x) { return fb_tanhf(x); }
    static __device__ __forceinline__ float atanh(float x) { return fb_atanhf(x); }
    // clamp-free forms for lanes known to be inside the open intervals (same bits as the full functions there)
    static __device__ __forceinline__ float phi4_open(float x) {
        float e = fb_expf_core(x);
        float sp = (x > FB_SOFTPLUS_THR) ? x : fb_log1pf_ge1(e);
        return FB_SUB(sp, fb_logf(FB_SUB(e, 1.0f)));
    }
    static __device__ __forceinline__ float phi2_open(float x) {
        float e = fb_expf_core(x);
        return FB_SUB(fb_logf(FB_ADD(e, 1.0f)), fb_logf(FB_SUB(e, 1.0f)));
    }
    static __device__ __forceinline__ float logaddexp_open(float mx, float d) {      // d = mn - mx >= -17.5
        const float t = fb_expf_core(d);
        return FB_ADD(fb_logf(FB_ADD(1.0f, t)), mx);
    }
};

struct MathSfu {
    static constexpr bool kSharedVnCorr = true;        // fb_math.h fb_sfu_vn_corr: one correction term per side and variable
    static __device__ __forceinline__ float softplus(float x) { return fb_sfu_softplusf(x); }
    static __device__ __forceinline__ float logaddexp(float a, float b) { return fb_sfu_logaddexpf(a, b); }
    static __device__ __forceinline__ float phi4(float x) { return fb_sfu_phi4f(x); }
    static __device__ __forceinline__ float phi2(float x) { return fb_sfu_phi2f(x); }
    static __device__ __forceinline__ float tanh(float x) { return fb_sfu_tanhf(x); }
    static __device__ __forceinline__ float atanh(float x) { return fb_sfu_atanhf(x); }
    static __device__ __forceinline__ float phi4_open(float x) { return fb_sfu_phi4_open(x); }
    static __device__ __forceinline__ float phi2_open(float x) { return fb_sfu_phi2_open(x); }
    static __device__ __forceinline__ float logaddexp_open(float mx, float d) { return fb_sfu_logaddexp_open(mx, d); }
    // issue-bound: the independent FP32 operations of the hot loops go two per instruction (fb_math.h paired forms)
    static constexpr bool kPaired = true;
    static __device__ __forceinline__ float2 phi_open2(float2 x) { return fb_sfu_phi_open2(x); }
    static __device__ __forceinline__ float2 softplus2(float2 x) { return fb_sfu_softplusf2(x); }
    static __device__ __forceinline__ float2 logaddexp_open2(float2 mx, float2 d) { return fb_sfu_logaddexp_open2(mx, d); }
    static __device__ __forceinline__ float2 tanh2(float2 x) { return fb_sfu_tanhf2(x); }
};

// ------------------------------------------------------------------ saturated fast paths
// Value-dependent shortcuts that return exactly what the full evaluation returns:
//   phi(x) = phi(clip_hi) = +0          for x >= 16.635532,
//   phi(x) = phi(clip_lo) = 16.635532   for x <= 8.5e-8      (tests/test_math.py pins both), and
//   logaddexp(a, b) = 0 + max(a, b)     when min - max < -17.5 (exp < 2^-25, so 1 + exp rounds to 1
//                                        and log(1) = 0).
// Once a frame has converged nearly every message sits in these regimes; a warp whose lanes are all
// saturated skips the polynomial evaluation altogether (the vote only decides whether the full path
// is executed, never which value a lane takes).
// Inside a voted evaluation only the lanes with 8.5e-8 < x < 16.635532 keep the value: no clamp needed.
template <typename MATH, bool PHI4>
__device__ __forceinline__ float phi_eval(float x) { return PHI4 ? MATH::phi4_open(x) : MATH::phi2_open(x); }

template <typename MATH, bool PHI4>
__device__ __forceinline__ float phi_sat(float x) {
    const bool hi = x >= FB_PHI_CLIP_HI, lo = x <= FB_PHI_CLIP_LO;
    float r = hi ? 0.0f : FB_PHI_CLIP_HI;
    if (__any_sync(__activemask(), !(hi || lo))) {
        const float f = phi_eval<MATH, PHI4>(x);
        r = (hi || lo) ? r : f;
    }
    return r;
}

// G call sites under one vote: the G independent polynomial chains interleave (ILP) at the price of evaluating
// all G when any lane needs any of them.  Values are those of phi_sat.
template <typename MATH, bool PHI4, int G, bool FULL = false>
__device__ __forceinline__ void phi_sat_group(const float x[G], float r[G]) {
    bool sat[G], need = false;
#pragma unroll
    for (int k = 0; k < G; k++) {
        const bool hi = x[k] >= FB_PHI_CLIP_HI, lo = x[k] <= FB_PHI_CLIP_LO;
        sat[k] = hi || lo;
        r[k] = hi ? 0.0f : FB_PHI_CLIP_HI;
        need = need || !sat[k];
    }
    if (__any_sync(FULL ? 0xffffffffu : __activemask(), need)) {
        int k0 = 0;
        if constexpr (MATH::kPaired) {         // sites 2i, 2i+1 as one float2 evaluation (odd G: the last alone)
#pragma unroll
            for (; k0 + 1 < G; k0 += 2) {
                const float2 f = MATH::phi_open2(make_float2(x[k0], x[k0 + 1]));
                r[k0] = sat[k0] ? r[k0] : f.x;
                r[k0 + 1] = sat[k0 + 1] ? r[k0 + 1] : f.y;
            }
        }
#pragma unroll
        for (int k = k0; k < G; k++) {
            const float f = phi_eval<MATH, PHI4>(x[k]);
            r[k] = sat[k] ? r[k] : f;
        }
    }
}

template <typename MATH>
__device__ __forceinline__ float logaddexp_sat(float a, float b) {
    const float mx = fmaxf(a, b), mn = fminf(a, b);
    const bool sat = FB_SUB(mn, mx) < -17.5f;
    float r = FB_ADD(0.0f, mx);
    if (__any_sync(__activemask(), !sat)) {
        const float f = MATH::logaddexp_open(mx, FB_SUB(mn, mx));     // exp without its clamp: d >= -17.5 on the lanes that keep f
        r = sat ? r : f;
    }
    return r;
}

// G logaddexp sites under one vote (the warp is converged: full mask).  Values are those of logaddexp_sat.
template <typename MATH, int G>
__device__ __forceinline__ void logaddexp_sat_group(const float a[G], const float b[G], float r[G]) {
    float mx[G], d[G];
    bool need = false;
#pragma unroll
    for (int k = 0; k < G; k++) {
        mx[k] = fmaxf(a[k], b[k]);
        d[k] = FB_SUB(fminf(a[k], b[k]), mx[k]);
        r[k] = FB_ADD(0.0f, mx[k]);
        need = need || !(d[k] < -17.5f);
    }
    if (__any_sync(0xffffffffu, need)) {
#pragma unroll
        for (int k = 0; k < G; k++) {
            const float f = MATH::logaddexp_open(mx[k], d[k]);
            r[k] = (d[k] < -17.5f) ? r[k] : f;
        }
    }
}

// SFU arithmetic: the two edge-independent terms of a variable node's outgoing messages (fb_math.h fb_sfu_vn_corr), the x
// edges' (from lz, ly) and the z edges' (from lx, ly), evaluated under one warp vote.  PAIRED: the two as one float2
// evaluation (the regular fast path in paired arithmetic).
template <typename MATH, bool FULL, bool PAIRED = false>
__device__ __forceinline__ void vn_corr_pair(float lx, float ly, float lz, float &ux, float &cx, float &uz, float &cz) {
    ux = fminf(lz, ly); uz = fminf(lx, ly);
    float dx, dz;
    if constexpr (PAIRED) {
        const float2 d = FB_SUB2(make_float2(ly, ly), make_float2(lz, lx));
        dx = -fabsf(d.x); dz = -fabsf(d.y);
    } else {
        dx = -fabsf(FB_SUB(ly, lz)); dz = -fabsf(FB_SUB(ly, lx));
    }
    const bool satx = dx < -17.5f, satz = dz < -17.5f;
    cx = 0.0f; cz = 0.0f;
    if (__any_sync(FULL ? 0xffffffffu : __activemask(), !(satx && satz))) {
        float fx, fz;
        if constexpr (PAIRED) {
            const float2 f = MATH::logaddexp_open2(make_float2(0.0f, 0.0f), make_float2(dx, dz));
            fx = f.x; fz = f.y;
        } else {
            fx = MATH::logaddexp_open(0.0f, dx); fz = MATH::logaddexp_open(0.0f, dz);
        }
        cx = satx ? 0.0f : fx; cz = satz ? 0.0f : fz;
    }
}
__device__ __forceinline__ float vn_msg(float num, float a, float u, float corr) { return FB_SUB(num, FB_ADD(FB_SUB(a, u), corr)); }

// ------------------------------------------------------------------ check nodes -------
// Update one check node in place: msg[] holds v2c on entry, c2v on exit.  Two passes over
// the check's edges; pass 1 parks phi(|m|) in the message slot and the signs in a bit mask
// (check degree <= 64 is enforced when the graph is created).
template <bool PHI4, typename MATH>
__device__ __forceinline__ void cn_update_one(const idx_t *__restrict__ cn_edge, int k0, int k1,
                                              float *msg, int synd_bit, int cn_type, float factor) {
    if (cn_type == 0) {
        unsigned long long mask = 0ull;
        int par = synd_bit;
        float T = 0.0f;
        for (int k = k0; k < k1; k++) {
            const int e = cn_edge[k];
            const float m = msg[e];
            const int neg = m < 0.0f;
            mask |= (unsigned long long)neg << (k - k0);
            par ^= neg;
            const float a = phi_sat<MATH, PHI4>(fabsf(m));
            msg[e] = a;
            T = FB_ADD(T, a);
        }
        for (int k = k0; k < k1; k++) {
            const int e = cn_edge[k];
            const float x = FB_SUB(T, msg[e]);
            float v = phi_sat<MATH, PHI4>(x);
            const int s = par ^ (int)((mask >> (k - k0)) & 1ull);
            v = s ? -v : v;
            msg[e] = FB_MUL(v, factor);
        }
    } else if (cn_type == 1) {
        float P = 1.0f;
        for (int k = k0; k < k1; k++) {
            const int e = cn_edge[k];
            float t = MATH::tanh(FB_MUL(msg[e], 0.5f));
            if (t == 0.0f) t = 1e-12f;
            msg[e] = t;
            P = FB_MUL(P, t);
        }
        P = synd_bit ? -P : P;
        for (int k = k0; k < k1; k++) {
            const int e = cn_edge[k];
            float v = FB_MUL(FB_DIV(1.0f, msg[e]), P);
            if (fabsf(v) < 1e-7f) v = 0.0f;
            v = FB_FMIN(FB_FMAX(v, -FB_ATANH_CLIP), FB_ATANH_CLIP);
            v = FB_MUL(2.0f, MATH::atanh(v));
            msg[e] = FB_MUL(v, factor);
        }
    } else {
        const float LARGE = 10000.0f;
        unsigned long long mask = 0ull;
        int par = synd_bit;
        float mn = __int_as_float(0x7f800000);
        for (int k = k0; k < k1; k++) {
            const int e = cn_edge[k];
            float m = FB_FMIN(FB_FMAX(msg[e], -FB_LLR_MAX), FB_LLR_MAX);
            const int neg = m < 0.0f;
            mask |= (unsigned long long)neg << (k - k0);
            par ^= neg;
            const float a = fabsf(m);
            msg[e] = a;
            if (a < mn) mn = a;
        }
        float mn2 = __int_as_float(0x7f800000), sum = 0.0f;
        for (int k = k0; k < k1; k++) {
            const int e = cn_edge[k];
            float d = FB_SUB(msg[e], mn);
            if (d == 0.0f) d = LARGE;
            msg[e] = d;
            if (d < mn2) mn2 = d;
            sum = FB_ADD(sum, d);
        }
        mn2 = FB_ADD(mn2, mn);
        const float node_sum = FB_SUB(sum, 19999.0f);
        const float sg = (node_sum > 0.0f) ? 1.0f : ((node_sum < 0.0f) ? -1.0f : 0.0f);
        const float dm = FB_MUL(0.5f, FB_SUB(1.0f, sg));
        const float mne = FB_ADD(FB_MUL(FB_SUB(1.0f, dm), mn), FB_MUL(dm, mn2));
        for (int k = k0; k < k1; k++) {
            const int e = cn_edge[k];
            float v = (msg[e] == LARGE) ? mne : mn;
            const int s = par ^ (int)((mask >> (k - k0)) & 1ull);
            v = s ? -v : v;
            msg[e] = FB_MUL(v, factor);
        }
    }
}

// ------------------------------------------------------------------ regular fast path --
// (DV, DC)-regular sides (every variable in DV checks, every check on DC variables): the edge
// ranges are v*DV.. and c*DC.., all loops unroll, the phi values and signs of a check stay in
// registers and the DC (or 2*DV) independent phi / logaddexp chains give the scheduler ILP.
// Operation order is exactly that of the generic path (and of the oracle).
// `rec` (optional): per-variable record written by the preceding VN phase -- bit s set if the incoming
// c2v message in slot s (x edges 0..DV-1, z edges DV..2DV-1) was negative, bit 15 set unless all of them
// had the saturated magnitude phi_max * factor.  The function returns true iff every message it writes
// is bit-identical to the one it replaces (saturated magnitude, same sign): when that holds for all
// checks of a frame the decoder state is a fixed point of the (deterministic) iteration and the
// remaining iterations cannot change it.
// FULL: the caller guarantees that all 32 lanes of the warp are here (k_bp4 runs the whole warps of a node loop through
// this instantiation and the ragged last warp through the other one), so the votes use the full mask -- no activemask /
// divergence check around each of them.
template <int DC, int DV, bool PHI4, typename MATH, bool FPX, bool FULL = false>
__device__ __forceinline__ bool cn_phi_regular(const idx_t *__restrict__ cn_edge, int c, float *msg,
                                               int synd_bit, float factor, const uint16_t *rec, int slot0) {
    int e[DC];
    float a[DC];
    // Signs.  The quaternary decoder's variable-to-check messages are differences num - logaddexp(..) of this kernel's own
    // making: never -0.0 (x - y rounds to +0 when it is zero) and never NaN, so "m < 0" IS the sign bit and the parity
    // of the signs is an XOR of the message words (SIGNBITS).  The binary decoder keeps the comparisons: its messages
    // can be scaled by negative edge weights, which makes -0.0 reachable, and sign(-0.0) counts as +1 in the reference.
    constexpr bool SIGNBITS = PHI4;
    uint32_t neg = 0, word[DC], pw = (uint32_t)synd_bit << 31;
    int par = synd_bit;
#pragma unroll
    for (int k = 0; k < DC; k++) e[k] = cn_edge[c * DC + k];
    // phi call sites evaluated under one warp vote: the GRP polynomial chains interleave (the single-site form leaves the
    // warp latency-bound on one Horner chain).  Measured on B200 (profiles/r02_lab_k_bp4_variants.txt, headline
    // pipeline): group 1 / 2 / 3 / 6 = 184.0 / 188.2 / 189.3 / 185.0 k frames/s.
    constexpr int GRP = DC % 3 == 0 ? 3 : (DC % 2 == 0 ? 2 : 1);
    float xin[DC];
#pragma unroll
    for (int k = 0; k < DC; k++) {
        const float m = msg[e[k]];
        if (SIGNBITS) {
            word[k] = (uint32_t)__float_as_int(m);
            pw ^= word[k];
        } else {
            const uint32_t sgn = (m < 0.0f) ? 1u : 0u;
            neg |= sgn << k;
            par ^= (int)sgn;
        }
        xin[k] = fabsf(m);
    }
    pw &= 0x80000000u;                              // parity of the signs and the syndrome bit, in the sign position
#pragma unroll
    for (int k = 0; k < DC; k += GRP) phi_sat_group<MATH, PHI4, GRP, FULL>(xin + k, a + k);
    float T = 0.0f;
#pragma unroll
    for (int k = 0; k < DC; k++) T = FB_ADD(T, a[k]);
    bool stable = FPX && rec != nullptr;
    float xo[DC], vo[DC];
    constexpr int NP = MATH::kPaired ? DC / 2 : 0;  // sites 2i, 2i+1 paired (odd DC: the last alone)
#pragma unroll
    for (int i = 0; i < NP; i++) {
        const float2 x2 = FB_SUB2(make_float2(T, T), make_float2(a[2 * i], a[2 * i + 1]));
        xo[2 * i] = x2.x; xo[2 * i + 1] = x2.y;
    }
#pragma unroll
    for (int k = 2 * NP; k < DC; k++) xo[k] = FB_SUB(T, a[k]);
#pragma unroll
    for (int k = 0; k < DC; k += GRP) phi_sat_group<MATH, PHI4, GRP, FULL>(xo + k, vo + k);
    bool allsat = true;
    uint32_t sw[DC];                                // sign of the outgoing message, in the sign position
    float v[DC];
#pragma unroll
    for (int k = 0; k < DC; k++) {
        sw[k] = SIGNBITS ? ((word[k] & 0x80000000u) ^ pw) : ((((uint32_t)par ^ (neg >> k)) & 1u) << 31);
        v[k] = __int_as_float(__float_as_int(vo[k]) ^ (int)sw[k]);
        allsat = allsat && (xo[k] <= FB_PHI_CLIP_LO);
        if (k < 2 * NP && (k & 1)) {
            const float2 m2 = FB_MUL2(make_float2(v[k - 1], v[k]), make_float2(factor, factor));
            msg[e[k - 1]] = m2.x; msg[e[k]] = m2.y;
        } else if (k >= 2 * NP) {
            msg[e[k]] = FB_MUL(v[k], factor);
        }
    }
    if (FPX && rec) {
        // one vote per check: only the AND over the whole frame is used (k_bp4's __syncthreads_and), so a warp with
        // any unsaturated output skips the record look-ups of all its lanes
        if (__all_sync(FULL ? 0xffffffffu : __activemask(), allsat)) {
#pragma unroll
            for (int k = 0; k < DC; k++) {
                const int vv = e[k] / DV;
                const int r = rec[vv];
                stable = stable && !(r & 0x8000) && ((uint32_t)((r >> (e[k] - vv * DV + slot0)) & 1) == (sw[k] >> 31));
            }
        } else {
            stable = false;
        }
    }
    return stable;
}

template <int DV, typename MATH, bool FPX, bool FULL = false>
__device__ __forceinline__ void vn_update_regular(int v, float *mx, float *mz, float px, float py, float pz,
                                                  uint16_t *rec, int sat_bits) {
    float ax[DV], az[DV];
#pragma unroll
    for (int k = 0; k < DV; k++) {
        ax[k] = mx[v * DV + k];
        az[k] = mz[v * DV + k];
    }
    if (FPX && rec) {      // signs of the incoming messages and whether all of them are saturated (see cn_phi_regular)
        int r = 0, bad = 0;
#pragma unroll
        for (int k = 0; k < DV; k++) {
            const int bx = __float_as_int(ax[k]), bz = __float_as_int(az[k]);
            r |= ((bx >> 31) & 1) << k;
            r |= ((bz >> 31) & 1) << (DV + k);
            bad |= ((bx & 0x7fffffff) ^ sat_bits) | ((bz & 0x7fffffff) ^ sat_bits);
        }
        rec[v] = (uint16_t)(bad ? 0x8000 : r);
    }
    if constexpr (MATH::kPaired && MATH::kSharedVnCorr) {
        // lane x: the x edges' chain, lane y: the z edges' -- the two sums keep their order, each message is vn_msg
        float2 S = make_float2(0.0f, 0.0f);
#pragma unroll
        for (int k = 0; k < DV; k++) S = FB_ADD2(S, make_float2(ax[k], az[k]));
        const float ly = FB_ADD(FB_ADD(S.y, S.x), py);
        const float2 l = FB_ADD2(make_float2(S.y, S.x), make_float2(px, pz));         // (lx, lz)
        const float2 num = MATH::softplus2(fb2_neg(l));
        float ux, cx, uz, cz;
        vn_corr_pair<MATH, FULL, true>(l.x, ly, l.y, ux, cx, uz, cz);
#pragma unroll
        for (int k = 0; k < DV; k++) {
            const float2 m = fb_sfu_vn_msg2(num, make_float2(ax[k], az[k]), make_float2(ux, uz), make_float2(cx, cz));
            mx[v * DV + k] = m.x;
            mz[v * DV + k] = m.y;
        }
        return;
    }
    float Sx = 0.0f, Sz = 0.0f;
#pragma unroll
    for (int k = 0; k < DV; k++) Sx = FB_ADD(Sx, ax[k]);
#pragma unroll
    for (int k = 0; k < DV; k++) Sz = FB_ADD(Sz, az[k]);
    const float ly = FB_ADD(FB_ADD(Sz, Sx), py);
    const float lx = FB_ADD(Sz, px);
    const float lz = FB_ADD(Sx, pz);
    const float num_hx = MATH::softplus(-lx), num_hz = MATH::softplus(-lz);
    if (MATH::kSharedVnCorr) {
        float ux, cx, uz, cz;
        vn_corr_pair<MATH, FULL>(lx, ly, lz, ux, cx, uz, cz);
#pragma unroll
        for (int k = 0; k < DV; k++) {
            mx[v * DV + k] = vn_msg(num_hx, ax[k], ux, cx);
            mz[v * DV + k] = vn_msg(num_hz, az[k], uz, cz);
        }
        return;
    }
    if (FULL) {
        // the 2 DV logaddexp sites under votes of 3 sites if 3 divides 2 DV, else of DV sites (same values as one vote per
        // site).  Measured on B200 when the SFU arithmetic still took this path (profiles/r02_lab_k_bp4_variants.txt):
        // groups of 3 / 6 / 2 = 316.4 / 312.5 / 315.4 k frames/s.
        constexpr int LG = (2 * DV) % 3 == 0 ? 3 : DV;
        float p[2 * DV], q[2 * DV], r[2 * DV];
#pragma unroll
        for (int k = 0; k < DV; k++) {
            p[k] = -FB_SUB(lz, ax[k]); q[k] = -FB_SUB(ly, ax[k]);
            p[DV + k] = -FB_SUB(lx, az[k]); q[DV + k] = -FB_SUB(ly, az[k]);
        }
#pragma unroll
        for (int k = 0; k < 2 * DV; k += LG) logaddexp_sat_group<MATH, LG>(p + k, q + k, r + k);
#pragma unroll
        for (int k = 0; k < DV; k++) {
            mx[v * DV + k] = FB_SUB(num_hx, r[k]);
            mz[v * DV + k] = FB_SUB(num_hz, r[DV + k]);
        }
        return;
    }
#pragma unroll
    for (int k = 0; k < DV; k++)
        mx[v * DV + k] = FB_SUB(num_hx, logaddexp_sat<MATH>(-FB_SUB(lz, ax[k]), -FB_SUB(ly, ax[k])));
#pragma unroll
    for (int k = 0; k < DV; k++)
        mz[v * DV + k] = FB_SUB(num_hz, logaddexp_sat<MATH>(-FB_SUB(lx, az[k]), -FB_SUB(ly, az[k])));
}

// ------------------------------------------------------------------ bulk-async staging --
// TMA 1-D bulk copies (cp.async.bulk, SASS UBLKCP): one thread posts the transfers against an mbarrier, nobody spends
// load / store instructions on them.  Source, destination and size must be multiples of 16 bytes.
__device__ __forceinline__ uint32_t bulk_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bulk_mbar_init(uint64_t *bar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bulk_smem_u32(bar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void bulk_expect(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bulk_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    constexpr uint32_t CHUNK = 32768;
    for (uint32_t off = 0; off < bytes; off += CHUNK)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(bulk_smem_u32(dst) + off), "l"(reinterpret_cast<const char *>(src) + off),
                        "r"(min(CHUNK, bytes - off)), "r"(bulk_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bulk_smem_u32(bar)), "r"(parity) : "memory");
    } while (!ok);
}
__host__ __device__ inline int pad4(int x) { return (x + 3) & ~3; }
__host__ __device__ inline int pad16(int x) { return (x + 15) & ~15; }

// ------------------------------------------------------------------ quaternary BP -----
struct Bp4Args {
    SideDev X, Z;
    int cn_type, num_iter;
    float factor;
    const int *frame_list;              // optional: CTA i decodes frame frame_list[i]
    View3<const float> llr;             // (b, k, v); ptr == nullptr -> constant prior
    float prior;
    View2<const uint8_t> sx, sz;        // (c, b)
    // pipeline workspace layout (optional, set together with llr / sx / sz): frame b's priors are the contiguous block
    // llr_bulk + b * 3 * pad4(n) ([3][pad4(n)] floats) and its syndrome bytes synd_bulk + b * pad16(m_x + m_z) -- both 16-byte
    // aligned, so the prologue stages them with bulk-async (TMA) copies instead of per-element loads
    const float *llr_bulk;
    const uint8_t *synd_bulk;
    View2<float> Lx, Ly, Lz;            // (b, v)   optional
    View2<uint8_t> xh, zh;              // (b, v)   optional (layer mode)
    View2<float> xl, zl;                // (row, b) optional: x_logit over hz rows, z_logit over hx rows
    View2<float> msg_x, msg_z;          // (b, e)   optional dump of the final c2v messages
    View3<float> iter_logits;           // (slot, row, b) optional: soft syndromes before every iteration and after
                                        // the last (slot 2*it = x_logit, 2*it+1 = z_logit; decoding_q.py:743-746)
    // pipeline mode (vbits != nullptr): decision + activity bookkeeping of feedback_gnn.py:322-340
    uint8_t *vbits;                     // [B][n], bits 2,3 receive the decision of active frames
    const uint8_t *active_in;           // [B] or nullptr (= all active)
    uint8_t *active_out;                // [B]
    uint8_t *rounds;                    // [B] incremented when the frame stays active (or nullptr)
    int *next_list, *next_count;        // optional compaction of still-active frames
    uint8_t *iters_out;                 // optional [B]: OPT-IN early stop (SURVEY.md H8; not what the reference does) -- a
                                        // frame leaves the loop once its hard decision reproduces the syndrome (warp-ballot
                                        // check after every iteration); iters_out[b] = iterations executed
    // optional row sets of the soft syndromes (CSR, int ptr / u16 col): the dense hx_perp / hz_perp rows of the reference's
    // trainable mode (decoding_q.py:32-37, 93-94); default = rows of hz (x_logit) and hx (z_logit)
    const int *rows_x_ptr, *rows_z_ptr;
    const idx_t *rows_x_col, *rows_z_col;
    int rows_x_m, rows_z_m;
    unsigned long long *stats;          // optional [2]: += {frames decoded, BP iterations actually executed} (bench.py's
                                        // executed-work roofline; the fixed-point exit skips iterations)
    float *state;                       // GSTATE kernels: per-CTA message / prior arrays in HBM (codes beyond shared memory)
    int64_t state_stride;               // floats per CTA
};

// Soft syndromes of the current message state (stage_two / trainable output of the reference):
// marginals from the messages, llr_x' / llr_z', then per check row sign * phi(sum phi(|.|)).
// scr: 2n floats of scratch, sgn: n bytes.  Generic (CSR) loops; not on the evaluation hot path.
template <bool CONST_PRIOR, typename MATH>
__device__ void bp4_iter_logits(const Bp4Args &a, const float *mx, const float *mz, const float *pri,
                                float *scr, uint8_t *sgn, int64_t b, int slot) {
    const SideDev &X = a.X, &Z = a.Z;
    const int n = X.n, T = blockDim.x, tid = threadIdx.x;
    for (int v = tid; v < n; v += T) {
        float Sx = 0.0f, Sz = 0.0f;
        for (int e = X.vn_ptr[v]; e < X.vn_ptr[v + 1]; e++) Sx = FB_ADD(Sx, mx[e]);
        for (int e = Z.vn_ptr[v]; e < Z.vn_ptr[v + 1]; e++) Sz = FB_ADD(Sz, mz[e]);
        const int np = pad4(n);
        const float px = CONST_PRIOR ? a.prior : pri[v];
        const float py = CONST_PRIOR ? a.prior : pri[np + v];
        const float pz = CONST_PRIOR ? a.prior : pri[2 * np + v];
        const float ly = FB_ADD(FB_ADD(Sz, Sx), py);
        const float lx = FB_ADD(Sz, px);
        const float lz = FB_ADD(Sx, pz);
        const float llr_zp = FB_SUB(MATH::softplus(-lx), MATH::logaddexp(-lz, -ly));
        const float llr_xp = FB_SUB(MATH::softplus(-lz), MATH::logaddexp(-lx, -ly));
        sgn[v] = (uint8_t)(((llr_xp < 0.0f) ? 1 : 0) | ((llr_zp < 0.0f) ? 2 : 0));
        scr[v] = MATH::phi4(fabsf(llr_xp));
        scr[n + v] = MATH::phi4(fabsf(llr_zp));
    }
    __syncthreads();
    if (a.rows_x_ptr) {                                 // custom row sets (dense hx_perp / hz_perp of the trainable mode)
        for (int c = tid; c < a.rows_x_m + a.rows_z_m; c += T) {
            const bool isz = c >= a.rows_x_m;           // rows_z -> z_logit (from llr_z'), rows_x -> x_logit
            const int cc = isz ? c - a.rows_x_m : c;
            const int *ptr = isz ? a.rows_z_ptr : a.rows_x_ptr;
            const idx_t *col = isz ? a.rows_z_col : a.rows_x_col;
            const float *sc = isz ? scr + n : scr;
            int par = 0;
            float Tsum = 0.0f;
            for (int k = ptr[cc]; k < ptr[cc + 1]; k++) {
                const int v = col[k];
                par ^= (sgn[v] >> (isz ? 1 : 0)) & 1;
                Tsum = FB_ADD(Tsum, sc[v]);
            }
            float val = MATH::phi4(Tsum);
            val = par ? -val : val;
            a.iter_logits(2 * slot + (isz ? 1 : 0), cc, b) = val;
        }
        __syncthreads();
        return;
    }
    for (int c = tid; c < X.m + Z.m; c += T) {
        const bool isx = c < X.m;                       // hx row -> z_logit (from llr_z'), hz row -> x_logit
        const SideDev &S = isx ? X : Z;
        const int cc = isx ? c : c - X.m;
        const float *sc = isx ? scr + n : scr;
        int par = 0;
        float Tsum = 0.0f;
        for (int k = S.cn_ptr[cc]; k < S.cn_ptr[cc + 1]; k++) {
            const int v = S.cn_vn[k];
            par ^= (sgn[v] >> (isx ? 1 : 0)) & 1;
            Tsum = FB_ADD(Tsum, sc[v]);
        }
        float val = MATH::phi4(Tsum);
        val = par ? -val : val;
        a.iter_logits(2 * slot + (isx ? 1 : 0), cc, b) = val;
    }
    __syncthreads();
}

// One CTA decodes one frame.  Dynamic shared memory (np = pad4(n), mp = pad16(m_x + m_z); every float block starts on a
// 16-byte boundary so the per-frame inputs can arrive by bulk-async copies):
//   float pri[(CONST_PRIOR ? 2 : 3) * np];  u8 sb[mp] (sbx then sbz);  float msg_x[E_x], msg_z[E_z], (scr[2 np] if
//   iter_logits);  u16 rec[n];  u8 dec[n]
// GSTATE (codes whose state exceeds the 227 KB of an SM): the float arrays live in the CTA's slice of an HBM
// scratch buffer (L2-resident while the CTA runs) instead; same code, same arithmetic, same results.
// Paired arithmetic on (3,6) / (4,8) codes: at least 2 CTAs of 512 threads, i.e. up to 64 registers.  Left alone, ptxas
// aims at 3 CTAs of 512 (40 registers), where the paired regular path spills.  On [[1270,28]] the launcher runs 256
// threads per CTA and shared memory allows 4 CTAs per SM, which 64 registers still allow (4 x 256 x 64 = 65 536).
// (5,10) needs more than 64 registers and keeps ptxas's choice.
template <bool CONST_PRIOR, int DV, int DC, typename MATH, bool FPX, bool GSTATE = false>
static __global__ void __launch_bounds__(512, (MATH::kPaired && DV > 0 && DV <= 4) ? 2 : 0) k_bp4(const Bp4Args a) {
    extern __shared__ __align__(16) float smem[];
    __shared__ __align__(8) uint64_t load_bar;
    const SideDev &X = a.X, &Z = a.Z;
    const int n = X.n, T = blockDim.x, tid = threadIdx.x;
    const int np = pad4(n), mp = pad16(X.m + Z.m), PRI = (CONST_PRIOR ? 2 : 3) * np;
    const int64_t b = a.frame_list ? a.frame_list[blockIdx.x] : blockIdx.x;
    float *gs = GSTATE ? a.state + (int64_t)blockIdx.x * a.state_stride : nullptr;
    float *pri = GSTATE ? gs : smem;
    uint8_t *sbx = GSTATE ? (uint8_t *)smem : (uint8_t *)(smem + PRI), *sbz = sbx + X.m;
    float *mx = GSTATE ? gs + PRI : (float *)(sbx + mp);
    float *mz = mx + X.E, *scr2 = mz + Z.E;
    uint16_t *rec = GSTATE ? (uint16_t *)(sbx + mp) : (uint16_t *)(scr2 + (a.iter_logits.ptr ? 2 * np : 0));
    uint8_t *dec = (uint8_t *)(rec + ((n + 1) & ~1));
    const idx_t *cn_edge_x = X.cn_edge, *cn_edge_z = Z.cn_edge;

    // per-frame inputs: the pipeline's workspace rows are 16-byte aligned blocks -> two bulk-async (TMA) copies posted by one
    // thread, overlapped with the clearing of the messages; the layer API's strided views are read element by element
    const bool bulk_pri = !GSTATE && !CONST_PRIOR && a.llr_bulk != nullptr;
    const bool bulk_syn = !GSTATE && a.synd_bulk != nullptr;
    if (bulk_pri || bulk_syn) {
        if (tid == 0) bulk_mbar_init(&load_bar);
        __syncthreads();
        if (tid == 0) {
            const uint32_t bytes = (bulk_pri ? (uint32_t)PRI * 4u : 0u) + (bulk_syn ? (uint32_t)mp : 0u);
            bulk_expect(&load_bar, bytes);
            if (bulk_pri) bulk_g2s(pri, a.llr_bulk + b * PRI, (uint32_t)PRI * 4u, &load_bar);
            if (bulk_syn) bulk_g2s(sbx, a.synd_bulk + b * mp, (uint32_t)mp, &load_bar);
        }
    }
    for (int e = tid; e < X.E + Z.E; e += T) mx[e] = 0.0f;
    if (!CONST_PRIOR && !bulk_pri)
        for (int k = 0; k < 3; k++)
            for (int v = tid; v < n; v += T) pri[k * np + v] = a.llr(b, k, v);
    if (!bulk_syn) {
        for (int c = tid; c < X.m; c += T) sbx[c] = a.sx(c, b);
        for (int c = tid; c < Z.m; c += T) sbz[c] = a.sz(c, b);
    }
    if (bulk_pri || bulk_syn) bulk_wait(&load_bar, 0);
    __syncthreads();

    const bool fast = DV > 0 && a.cn_type == 0;     // regular graph + boxplus-phi: unrolled path
    // Fixed-point exit: once an iteration reproduces every message bit for bit
    // the remaining iterations are no-ops, so they are skipped -- the outputs are unchanged by construction.
    // Only worth its bookkeeping for long runs (the 64-iteration first stage), and never before iteration 6.
    const bool fp_exit = FPX && fast && !a.iter_logits.ptr;
    const int sat_bits = __float_as_int(FB_MUL(FB_PHI_CLIP_HI, a.factor)) & 0x7fffffff;   // |phi(clip_lo) * factor|
    int it_done = a.num_iter;
    for (int it = 0; it < a.num_iter; it++) {
        if (a.iter_logits.ptr) bp4_iter_logits<CONST_PRIOR, MATH>(a, mx, mz, pri, scr2, dec, b, it);
        // the fixed-point test runs every third iteration: a later test only delays the exit by no-op iterations.  Measured
        // on B200 (profiles/r02_lab_k_bp4_variants.txt): stride 1 / 2 / 3 / 4 = 414 / 434 / 441 / 436 k frames/s.
        uint16_t *recp = (fp_exit && it >= 6 && (it % 3) == 0) ? rec : nullptr;
        // variable nodes (decoding_q.py:227-275)
        if (DV > 0) {
            // whole warps take the full-mask instantiation, the ragged last warp the activemask one (the launchers only use
            // multiples of 32 threads)
            for (int v = tid; v < n; v += T) {
                const float px = CONST_PRIOR ? a.prior : pri[v];
                const float py = CONST_PRIOR ? a.prior : pri[np + v];
                const float pz = CONST_PRIOR ? a.prior : pri[2 * np + v];
                if ((v | 31) < n) vn_update_regular<(DV > 0 ? DV : 1), MATH, FPX, true>(v, mx, mz, px, py, pz, recp, sat_bits);
                else vn_update_regular<(DV > 0 ? DV : 1), MATH, FPX, false>(v, mx, mz, px, py, pz, recp, sat_bits);
            }
        } else
        for (int v = tid; v < n; v += T) {
            const float px = CONST_PRIOR ? a.prior : pri[v];
            const float py = CONST_PRIOR ? a.prior : pri[np + v];
            const float pz = CONST_PRIOR ? a.prior : pri[2 * np + v];
            const int x0 = X.vn_ptr[v], x1 = X.vn_ptr[v + 1], z0 = Z.vn_ptr[v], z1 = Z.vn_ptr[v + 1];
            float Sx = 0.0f, Sz = 0.0f;
            for (int e = x0; e < x1; e++) Sx = FB_ADD(Sx, mx[e]);
            for (int e = z0; e < z1; e++) Sz = FB_ADD(Sz, mz[e]);
            const float ly = FB_ADD(FB_ADD(Sz, Sx), py);
            const float lx = FB_ADD(Sz, px);
            const float lz = FB_ADD(Sx, pz);
            const float num_hx = MATH::softplus(-lx), num_hz = MATH::softplus(-lz);
            if (MATH::kSharedVnCorr) {
                float ux, cx, uz, cz;
                vn_corr_pair<MATH, false>(lx, ly, lz, ux, cx, uz, cz);
                for (int e = x0; e < x1; e++) mx[e] = vn_msg(num_hx, mx[e], ux, cx);
                for (int e = z0; e < z1; e++) mz[e] = vn_msg(num_hz, mz[e], uz, cz);
                continue;
            }
            for (int e = x0; e < x1; e++) {
                const float m = mx[e];
                mx[e] = FB_SUB(num_hx, logaddexp_sat<MATH>(-FB_SUB(lz, m), -FB_SUB(ly, m)));
            }
            for (int e = z0; e < z1; e++) {
                const float m = mz[e];
                mz[e] = FB_SUB(num_hz, logaddexp_sat<MATH>(-FB_SUB(lx, m), -FB_SUB(ly, m)));
            }
        }
        __syncthreads();
        // check nodes of both sides as one index space
        bool stable = true;
        if (fast) {
            const int mt = X.m + Z.m;
            for (int c = tid; c < mt; c += T) {
                const bool isx = c < X.m;
                const int cc = isx ? c : c - X.m;
                if ((c | 31) < mt)
                    stable &= cn_phi_regular<(DC > 0 ? DC : 1), (DV > 0 ? DV : 1), true, MATH, FPX, true>(
                        isx ? cn_edge_x : cn_edge_z, cc, isx ? mx : mz, isx ? sbx[cc] : sbz[cc], a.factor, recp, isx ? 0 : DV);
                else
                    stable &= cn_phi_regular<(DC > 0 ? DC : 1), (DV > 0 ? DV : 1), true, MATH, FPX, false>(
                        isx ? cn_edge_x : cn_edge_z, cc, isx ? mx : mz, isx ? sbx[cc] : sbz[cc], a.factor, recp, isx ? 0 : DV);
            }
        } else
        for (int c = tid; c < X.m + Z.m; c += T) {
            const bool isx = c < X.m;
            const int cc = isx ? c : c - X.m;
            float *msg = isx ? mx : mz;
            const int sb = isx ? sbx[cc] : sbz[cc];
            const SideDev &S = isx ? X : Z;
            cn_update_one<true, MATH>(S.cn_edge, S.cn_ptr[cc], S.cn_ptr[cc + 1], msg, sb, a.cn_type, a.factor);
        }
        if (FPX && recp) {
            if (__syncthreads_and(stable)) { it_done = it + 1; break; }
        } else {
            __syncthreads();
        }
        if (a.iters_out) {
            // opt-in early stop: hard decision of the current messages, then the syndrome of that decision
            for (int v = tid; v < n; v += T) {
                float Sx = 0.0f, Sz = 0.0f;
                for (int e = X.vn_ptr[v]; e < X.vn_ptr[v + 1]; e++) Sx = FB_ADD(Sx, mx[e]);
                for (int e = Z.vn_ptr[v]; e < Z.vn_ptr[v + 1]; e++) Sz = FB_ADD(Sz, mz[e]);
                const float px = CONST_PRIOR ? a.prior : pri[v];
                const float py = CONST_PRIOR ? a.prior : pri[np + v];
                const float pz = CONST_PRIOR ? a.prior : pri[2 * np + v];
                const float ly = FB_ADD(FB_ADD(Sz, Sx), py), lx = FB_ADD(Sz, px), lz = FB_ADD(Sx, pz);
                int d = 0;
                float best = 0.0f;
                if (lx < best) { best = lx; d = 1; }
                if (lz < best) { best = lz; d = 2; }
                if (ly < best) { best = ly; d = 3; }
                dec[v] = (uint8_t)d;
            }
            __syncthreads();
            bool bad = false;
            const int mt = X.m + Z.m, mround = (mt + 31) & ~31;
            for (int c = tid; c < mround; c += T) {
                int par = 0;
                if (c < mt) {
                    const bool isx = c < X.m;                   // hx rows check z_hat (bit 1), hz rows check x_hat (bit 0)
                    const SideDev &S = isx ? X : Z;
                    const int cc = isx ? c : c - X.m;
                    par = isx ? sbx[cc] : sbz[cc];
                    for (int k = S.cn_ptr[cc]; k < S.cn_ptr[cc + 1]; k++) par ^= (dec[S.cn_vn[k]] >> (isx ? 1 : 0)) & 1;
                }
                bad |= __ballot_sync(0xffffffffu, par) != 0u;   // one vote per 32 checks
            }
            if (!__syncthreads_or(bad)) { it_done = it + 1; break; }
        }
    }

    if (a.stats && tid == 0) { atomicAdd(a.stats, 1ull); atomicAdd(a.stats + 1, (unsigned long long)it_done); }
    if (a.iters_out && tid == 0) a.iters_out[b] = (uint8_t)it_done;
    if (a.iter_logits.ptr) bp4_iter_logits<CONST_PRIOR, MATH>(a, mx, mz, pri, scr2, dec, b, a.num_iter);
    if (a.msg_x.ptr) for (int e = tid; e < X.E; e += T) a.msg_x(b, e) = mx[e];
    if (a.msg_z.ptr) for (int e = tid; e < Z.E; e += T) a.msg_z(b, e) = mz[e];

    // marginals, decision, per-variable terms of the soft syndromes (decoding_q.py:771-790,455-464)
    const bool want_logits = a.xl.ptr != nullptr || a.zl.ptr != nullptr;
    for (int v = tid; v < n; v += T) {
        float Sx = 0.0f, Sz = 0.0f;
        for (int e = X.vn_ptr[v]; e < X.vn_ptr[v + 1]; e++) Sx = FB_ADD(Sx, mx[e]);
        for (int e = Z.vn_ptr[v]; e < Z.vn_ptr[v + 1]; e++) Sz = FB_ADD(Sz, mz[e]);
        const float px = CONST_PRIOR ? a.prior : pri[v];
        const float py = CONST_PRIOR ? a.prior : pri[np + v];
        const float pz = CONST_PRIOR ? a.prior : pri[2 * np + v];
        const float ly = FB_ADD(FB_ADD(Sz, Sx), py);
        const float lx = FB_ADD(Sz, px);
        const float lz = FB_ADD(Sx, pz);
        if (a.Lx.ptr) a.Lx(b, v) = lx;
        if (a.Ly.ptr) a.Ly(b, v) = ly;
        if (a.Lz.ptr) a.Lz(b, v) = lz;
        int d = 0;
        float best = 0.0f;
        if (lx < best) { best = lx; d = 1; }
        if (lz < best) { best = lz; d = 2; }
        if (ly < best) { best = ly; d = 3; }
        if (want_logits) {
            const float llr_zp = FB_SUB(MATH::softplus(-lx), MATH::logaddexp(-lz, -ly));
            const float llr_xp = FB_SUB(MATH::softplus(-lz), MATH::logaddexp(-lx, -ly));
            d |= (llr_xp < 0.0f) << 2;
            d |= (llr_zp < 0.0f) << 3;
            pri[v] = MATH::phi4(fabsf(llr_xp));
            pri[np + v] = MATH::phi4(fabsf(llr_zp));
        }
        dec[v] = (uint8_t)d;
    }
    __syncthreads();

    // soft syndromes per check row and the syndrome match of the decision
    int mismatch = 0;
    for (int c = tid; c < X.m + Z.m; c += T) {
        const bool isx = c < X.m;                       // hx row: z_logit from llr_z', checks z_hat
        const SideDev &S = isx ? X : Z;
        const int cc = isx ? c : c - X.m;
        const float *scr = isx ? pri + np : pri;
        const int sbit = isx ? 3 : 2, dbit = isx ? 1 : 0;
        int par = 0, dpar = 0;
        float Tsum = 0.0f;
        for (int k = S.cn_ptr[cc]; k < S.cn_ptr[cc + 1]; k++) {
            const int v = S.cn_vn[k];
            const int dv = dec[v];
            par ^= (dv >> sbit) & 1;
            dpar ^= (dv >> dbit) & 1;
            if (want_logits) Tsum = FB_ADD(Tsum, scr[v]);
        }
        mismatch |= dpar ^ (isx ? sbx[cc] : sbz[cc]);
        if (want_logits && !a.rows_x_ptr) {
            float val = MATH::phi4(Tsum);
            val = par ? -val : val;
            if (isx) { if (a.zl.ptr) a.zl(cc, b) = val; }
            else     { if (a.xl.ptr) a.xl(cc, b) = val; }
        }
    }
    if (want_logits && a.rows_x_ptr) {
        for (int c = tid; c < a.rows_x_m + a.rows_z_m; c += T) {
            const bool isz = c >= a.rows_x_m;
            const int cc = isz ? c - a.rows_x_m : c;
            const int *ptr = isz ? a.rows_z_ptr : a.rows_x_ptr;
            const idx_t *col = isz ? a.rows_z_col : a.rows_x_col;
            const float *scr = isz ? pri + np : pri;
            int par = 0;
            float Tsum = 0.0f;
            for (int k = ptr[cc]; k < ptr[cc + 1]; k++) {
                const int v = col[k];
                par ^= (dec[v] >> (isz ? 3 : 2)) & 1;
                Tsum = FB_ADD(Tsum, scr[v]);
            }
            float val = MATH::phi4(Tsum);
            val = par ? -val : val;
            if (isz) { if (a.zl.ptr) a.zl(cc, b) = val; }
            else     { if (a.xl.ptr) a.xl(cc, b) = val; }
        }
    }
    if (a.xh.ptr) for (int v = tid; v < n; v += T) a.xh(b, v) = dec[v] & 1;
    if (a.zh.ptr) for (int v = tid; v < n; v += T) a.zh(b, v) = (dec[v] >> 1) & 1;
    if (a.vbits) {
        mismatch = __syncthreads_or(mismatch);
        const int act_in = a.active_in ? a.active_in[b] : 1;
        if (act_in) {
            uint8_t *vb = a.vbits + b * n;
            for (int v = tid; v < n; v += T) vb[v] = (vb[v] & 3) | ((dec[v] & 3) << 2);
        }
        if (tid == 0) {
            const int act_out = act_in && mismatch;
            a.active_out[b] = (uint8_t)act_out;
            if (a.rounds && act_out) a.rounds[b] += 1;
            if (a.next_list && act_out) a.next_list[atomicAdd(a.next_count, 1)] = (int)b;
        }
    }
}

// ------------------------------------------------------------------ binary BP ---------
struct Bp2Args {
    SideDev S;
    int cn_type, num_iter;
    float factor;
    View2<const float> llr;             // (b, v) logits; ptr == nullptr -> constant llr_const
    float llr_const;
    View2<const uint8_t> synd;          // (c, b) optional
    View2<float> soft;                  // (b, v) optional
    View2<uint8_t> hard;                // (b, v) optional
    uint8_t *vbits;                     // optional [B][n]: the hard decision goes to bit 2 (pipeline mode)
    int *next_list, *next_count;        // optional: frames whose decision misses the syndrome (for OSD-0)
    const float *edge_w;                // optional [E], VN order: per-edge weights on the v2c messages (trainable decoder,
                                        // decoding.py:981-983)
    View2<const float> msg_in;          // optional (b, e): initial c2v messages (stateful decoder, decoding.py:947-953)
    View2<float> msg_out;               // optional (b, e): final c2v messages
};

// smem: float msg[E], llr[n]; u8 sb[m], dec[n].  (DV, DC) > 0: regular graph, unrolled (boxplus-phi only).
template <int DV, int DC, typename MATH>
static __global__ void __launch_bounds__(512) k_bp2(const Bp2Args a) {
    extern __shared__ float smem[];
    const SideDev &S = a.S;
    const int n = S.n, T = blockDim.x, tid = threadIdx.x;
    const int64_t b = blockIdx.x;
    float *msg = smem, *llr = msg + S.E;
    uint8_t *sb = (uint8_t *)(llr + n), *dec = sb + S.m;
    for (int e = tid; e < S.E; e += T) msg[e] = a.msg_in.ptr ? a.msg_in(b, e) : 0.0f;
    for (int v = tid; v < n; v += T) {
        float l = a.llr.ptr ? a.llr(b, v) : a.llr_const;
        l = FB_FMIN(FB_FMAX(l, -FB_LLR_MAX), FB_LLR_MAX);
        llr[v] = -l;
    }
    for (int c = tid; c < S.m; c += T) sb[c] = a.synd.ptr ? a.synd(c, b) : 0;
    __syncthreads();
    const bool fast = DV > 0 && a.cn_type == 0;
    for (int it = 0; it < a.num_iter; it++) {
        for (int v = tid; v < n; v += T) {
            if (DV > 0) {
                constexpr int D = DV > 0 ? DV : 1;
                float m[D];
#pragma unroll
                for (int k = 0; k < D; k++) m[k] = msg[v * D + k];
                float s = 0.0f;
#pragma unroll
                for (int k = 0; k < D; k++) s = FB_ADD(s, m[k]);
                s = FB_ADD(s, llr[v]);
#pragma unroll
                for (int k = 0; k < D; k++) {
                    float o = FB_SUB(s, m[k]);
                    if (a.edge_w) o = FB_MUL(o, a.edge_w[v * D + k]);
                    msg[v * D + k] = o;
                }
                continue;
            }
            const int e0 = S.vn_ptr[v], e1 = S.vn_ptr[v + 1];
            float s = 0.0f;
            for (int e = e0; e < e1; e++) s = FB_ADD(s, msg[e]);
            s = FB_ADD(s, llr[v]);
            for (int e = e0; e < e1; e++) {
                float o = FB_SUB(s, msg[e]);
                if (a.edge_w) o = FB_MUL(o, a.edge_w[e]);
                msg[e] = o;
            }
        }
        __syncthreads();
        for (int c = tid; c < S.m; c += T) {
            if (fast) cn_phi_regular<(DC > 0 ? DC : 1), (DV > 0 ? DV : 1), false, MATH, false>(S.cn_edge, c, msg, sb[c], a.factor, nullptr, 0);
            else cn_update_one<false, MATH>(S.cn_edge, S.cn_ptr[c], S.cn_ptr[c + 1], msg, sb[c], a.cn_type, a.factor);
        }
        __syncthreads();
    }
    if (a.msg_out.ptr) for (int e = tid; e < S.E; e += T) a.msg_out(b, e) = msg[e];
    for (int v = tid; v < n; v += T) {
        float s = 0.0f;
        for (int e = S.vn_ptr[v]; e < S.vn_ptr[v + 1]; e++) s = FB_ADD(s, msg[e]);
        const float x = -FB_ADD(llr[v], s);
        if (a.soft.ptr) a.soft(b, v) = x;
        if (a.hard.ptr) a.hard(b, v) = (uint8_t)(0.0f < x);
        if (a.vbits) a.vbits[b * n + v] = (uint8_t)((a.vbits[b * n + v] & 3) | ((0.0f < x) ? 4 : 0));
        dec[v] = (uint8_t)(0.0f < x);
    }
    if (a.next_list) {
        __syncthreads();
        int mismatch = 0;
        for (int c = tid; c < S.m; c += T) {
            int par = sb[c];
            for (int k = S.cn_ptr[c]; k < S.cn_ptr[c + 1]; k++) par ^= dec[S.cn_vn[k]];
            mismatch |= par;
        }
        mismatch = __syncthreads_or(mismatch);
        if (tid == 0 && mismatch) a.next_list[atomicAdd(a.next_count, 1)] = (int)b;
    }
}

// ------------------------------------------------------------------ feedback GNN ------
struct GnnArgs {
    SideDev X, Z;
    const float *weights;               // packed, see GnnLayout
    int act, reduce, use_bias;
    const int *frame_list;
    int64_t num_frames;                 // frames to process (list length or B)
    View3<const float> h_vn;            // (b, v, k)
    View2<const float> logit_hx, logit_hz;   // (row, b)
    View2<const uint8_t> sx, sz;        // (c, b)
    View3<float> out;                   // (b, v, k)
};

// packed weight layout (floats): each block padded to a multiple of 4 floats
template <int H, int M> struct GnnLayout {
    static constexpr int pad4(int x) { return (x + 3) & ~3; }
    static constexpr int W1x = 0;
    static constexpr int b1x = W1x + pad4(4 * H);
    static constexpr int W2x = b1x + pad4(H);
    static constexpr int b2x = W2x + pad4(H * M);
    static constexpr int W1z = b2x + pad4(M);
    static constexpr int b1z = W1z + pad4(4 * H);
    static constexpr int W2z = b1z + pad4(H);
    static constexpr int b2z = W2z + pad4(H * M);
    static constexpr int W3 = b2z + pad4(M);
    static constexpr int b3 = W3 + pad4((2 * M + 3) * H);
    static constexpr int W0 = b3 + pad4(H);
    static constexpr int b0 = W0 + pad4(H * 3);
    // first-layer rows once more, one float4 {w_cn, w_Lx, w_Ly, w_Lz} per hidden unit (one LDS.128 in the regular path)
    static constexpr int W1tx = b0 + pad4(3);
    static constexpr int W1tz = W1tx + 4 * H;
    static constexpr int total = W1tz + 4 * H;
};

template <typename MATH>
__device__ __forceinline__ float gnn_act(int act, float x) {
    if (act == 0) return MATH::tanh(x);
    if (act == 1) return x > 0.0f ? x : 0.0f;
    return x;
}

// Weights staged per CTA in shared memory and read as broadcast loads.  (Measured alternative:
// __constant__ memory through LDC is 19 % slower for this kernel -- higher load latency, same FFMA
// operand traffic.)  Packed fma.rn.f32x2 sustains only 0.77x the lanes/s of scalar FFMA on B200
// (tools/micro/ffma2_bench.cu), so it loses wherever the FP32 pipe is the limit -- this kernel, and
// the exact arithmetic (MathExact::kPaired = false).  It wins where instruction issue is the limit
// and the FP32 pipe has room: the SFU kernels (MathSfu::kPaired).
struct WSmem {
    const float *p;
    __device__ __forceinline__ float ld(int i) const { return p[i]; }
    __device__ __forceinline__ float4 ld4(int i) const { return *reinterpret_cast<const float4 *>(p + i); }
};

// One thread per (frame, variable node).  Messages of one side into the variable node are computed
// and reduced as in feedback_gnn.py:175-184; the arithmetic and its order are those of
// oracle/fbgnn_oracle.c (gnn_side).
//   FACT   : reduce_op "mean" / "sum" -- the linear output layer of the edge MLP is applied once to
//            the sum of the hidden activations over the node's edges (W2^T sum_e t_e + deg b2), which
//            removes deg-1 of every deg H x M products;  !FACT ("max" / "min"): per-edge messages.
//   DV > 0 : both sides are DV-regular -- the DV edges of a side are processed together, so the DV
//            tanh chains overlap;  DV == 0 : any degrees.
//   TANH_BIAS : compile-time specialisation of the shipped configuration (tanh, use_bias=True);
//            otherwise activation / bias are run-time switches.
// The two sides share ONE copy of the inner loop (side loop not unrolled) and the loop over hidden
// units is unrolled by two only: the hot loop body stays a few KB, inside the instruction cache.
// Requires H % 4 == 0 and M % 4 == 0.
template <int H, int M, int DV, bool TANH_BIAS, bool FACT, typename MATH>
__device__ __forceinline__ void gnn_body(const GnnArgs &a, const WSmem w) {
    typedef GnnLayout<H, M> Lay;
    static_assert(FACT || DV == 0, "the per-edge form is only built for the generic degree path");
    constexpr int NE = DV > 0 ? DV : 1;
    const int n = a.X.n;
    const int act = TANH_BIAS ? 0 : a.act;
    const bool use_bias = TANH_BIAS ? true : (a.use_bias != 0);
    const int64_t items = a.num_frames * n;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items;
         it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t fi = it / n;
        const int v = (int)(it - fi * n);
        const int64_t b = a.frame_list ? a.frame_list[fi] : fi;
        const float f1 = a.h_vn(b, v, 0), f2 = a.h_vn(b, v, 1), f3 = a.h_vn(b, v, 2);
        float in[2 * M + 3];
        if (FACT && DV > 0) {
            // Regular sides, mean / sum: the 2 * DV tanh chains of one hidden unit (both sides) are evaluated together,
            // so their MUFU / FMA latencies overlap; per side the operations and their order are those of the
            // one-side loop below (and of the oracle's gnn_side).
            float hcx[NE], hcz[NE], rx[M], rz[M];
#pragma unroll
            for (int k = 0; k < NE; k++) {
                const int cx = a.X.vn_cn[v * NE + k], cz = a.Z.vn_cn[v * NE + k];
                const float lx = a.logit_hx(cx, b), lz = a.logit_hz(cz, b);
                hcx[k] = a.sx(cx, b) ? -lx : lx;
                hcz[k] = a.sz(cz, b) ? -lz : lz;
            }
#pragma unroll
            for (int i = 0; i < M; i++) { rx[i] = 0.0f; rz[i] = 0.0f; }
#pragma unroll 1
            for (int j = 0; j < H; j++) {
                const float4 wx = w.ld4(Lay::W1tx + 4 * j), wz = w.ld4(Lay::W1tz + 4 * j);
                const float bx = w.ld(Lay::b1x + j), bz = w.ld(Lay::b1z + j);
                const float basex = FB_FMA(f3, wx.w, FB_FMA(f2, wx.z, FB_FMA(f1, wx.y, 0.0f)));
                const float basez = FB_FMA(f3, wz.w, FB_FMA(f2, wz.z, FB_FMA(f1, wz.y, 0.0f)));
                float tx[NE], tz[NE];
#pragma unroll
                for (int k = 0; k < NE; k++) {
                    tx[k] = FB_FMA(hcx[k], wx.x, basex);
                    tz[k] = FB_FMA(hcz[k], wz.x, basez);
                    if (use_bias) { tx[k] = FB_ADD(tx[k], bx); tz[k] = FB_ADD(tz[k], bz); }
                }
#pragma unroll
                for (int k = 0; k < NE; k++) { tx[k] = gnn_act<MATH>(act, tx[k]); tz[k] = gnn_act<MATH>(act, tz[k]); }
                float hsx = tx[0], hsz = tz[0];
#pragma unroll
                for (int k = 1; k < NE; k++) { hsx = FB_ADD(hsx, tx[k]); hsz = FB_ADD(hsz, tz[k]); }
#pragma unroll
                for (int i = 0; i < M; i += 4) {
                    const float4 ux = w.ld4(Lay::W2x + j * M + i), uz = w.ld4(Lay::W2z + j * M + i);
                    rx[i + 0] = FB_FMA(hsx, ux.x, rx[i + 0]); rx[i + 1] = FB_FMA(hsx, ux.y, rx[i + 1]);
                    rx[i + 2] = FB_FMA(hsx, ux.z, rx[i + 2]); rx[i + 3] = FB_FMA(hsx, ux.w, rx[i + 3]);
                    rz[i + 0] = FB_FMA(hsz, uz.x, rz[i + 0]); rz[i + 1] = FB_FMA(hsz, uz.y, rz[i + 1]);
                    rz[i + 2] = FB_FMA(hsz, uz.z, rz[i + 2]); rz[i + 3] = FB_FMA(hsz, uz.w, rz[i + 3]);
                }
            }
            const float dg = (float)NE;
#pragma unroll
            for (int i = 0; i < M; i++) {
                float qx = rx[i], qz = rz[i];
                if (a.reduce == 0) {
                    qx = FB_DIV(qx, dg); qz = FB_DIV(qz, dg);
                    if (use_bias) { qx = FB_ADD(qx, w.ld(Lay::b2x + i)); qz = FB_ADD(qz, w.ld(Lay::b2z + i)); }
                } else if (use_bias) {
                    qx = FB_FMA(dg, w.ld(Lay::b2x + i), qx); qz = FB_FMA(dg, w.ld(Lay::b2z + i), qz);
                }
                in[i] = qx; in[M + i] = qz;
            }
        } else
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
            const SideDev &S = side ? a.Z : a.X;
            const int oW1 = side ? Lay::W1z : Lay::W1x, ob1 = side ? Lay::b1z : Lay::b1x;
            const int oW2 = side ? Lay::W2z : Lay::W2x, ob2 = side ? Lay::b2z : Lay::b2x;
            const View2<const float> &logit = side ? a.logit_hz : a.logit_hx;
            const View2<const uint8_t> &synd = side ? a.sz : a.sx;
            const int e0 = S.vn_ptr[v], e1 = S.vn_ptr[v + 1];
            float red[M];
#pragma unroll
            for (int i = 0; i < M; i++) red[i] = 0.0f;
            if (FACT) {
#pragma unroll 2
                for (int j = 0; j < H; j++) {
                    // features [h_cn, Lx, Ly, Lz]: the per-variable terms first, the check term last
                    const float base = FB_FMA(f3, w.ld(oW1 + 3 * H + j),
                                              FB_FMA(f2, w.ld(oW1 + 2 * H + j), FB_FMA(f1, w.ld(oW1 + H + j), 0.0f)));
                    const float w0 = w.ld(oW1 + j), bj = w.ld(ob1 + j);
                    float hs = 0.0f;
                    for (int e = e0; e < e1; e++) {
                        const int c = S.vn_cn[e];
                        const float lg = logit(c, b);
                        float t = FB_FMA(synd(c, b) ? -lg : lg, w0, base);
                        if (use_bias) t = FB_ADD(t, bj);
                        const float hv = gnn_act<MATH>(act, t);
                        hs = (e == e0) ? hv : FB_ADD(hs, hv);
                    }
#pragma unroll
                    for (int i = 0; i < M; i += 4) {
                        const float4 wv = w.ld4(oW2 + j * M + i);
                        red[i + 0] = FB_FMA(hs, wv.x, red[i + 0]);
                        red[i + 1] = FB_FMA(hs, wv.y, red[i + 1]);
                        red[i + 2] = FB_FMA(hs, wv.z, red[i + 2]);
                        red[i + 3] = FB_FMA(hs, wv.w, red[i + 3]);
                    }
                }
                const float dg = (float)(e1 - e0);
#pragma unroll
                for (int i = 0; i < M; i++) {
                    float r = red[i];
                    if (a.reduce == 0) {
                        r = FB_DIV(r, dg);
                        if (use_bias) r = FB_ADD(r, w.ld(ob2 + i));
                    } else if (use_bias) {
                        r = FB_FMA(dg, w.ld(ob2 + i), r);
                    }
                    red[i] = (e1 > e0) ? r : 0.0f;
                }
            } else {
                for (int e = e0; e < e1; e++) {
                    const int c = S.vn_cn[e];
                    const float lg = logit(c, b);
                    const float hc = synd(c, b) ? -lg : lg;
                    float acc[M];
#pragma unroll
                    for (int i = 0; i < M; i++) acc[i] = 0.0f;
#pragma unroll 2
                    for (int j = 0; j < H; j++) {
                        const float base = FB_FMA(f3, w.ld(oW1 + 3 * H + j),
                                                  FB_FMA(f2, w.ld(oW1 + 2 * H + j), FB_FMA(f1, w.ld(oW1 + H + j), 0.0f)));
                        float t = FB_FMA(hc, w.ld(oW1 + j), base);
                        if (use_bias) t = FB_ADD(t, w.ld(ob1 + j));
                        const float hv = gnn_act<MATH>(act, t);
#pragma unroll
                        for (int i = 0; i < M; i += 4) {
                            const float4 wv = w.ld4(oW2 + j * M + i);
                            acc[i + 0] = FB_FMA(hv, wv.x, acc[i + 0]);
                            acc[i + 1] = FB_FMA(hv, wv.y, acc[i + 1]);
                            acc[i + 2] = FB_FMA(hv, wv.z, acc[i + 2]);
                            acc[i + 3] = FB_FMA(hv, wv.w, acc[i + 3]);
                        }
                    }
#pragma unroll
                    for (int i = 0; i < M; i++) {
                        const float mval = use_bias ? FB_ADD(acc[i], w.ld(ob2 + i)) : acc[i];
                        if (e == e0) red[i] = mval;
                        else if (a.reduce == 2) red[i] = (mval > red[i]) ? mval : red[i];
                        else red[i] = (mval < red[i]) ? mval : red[i];
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < M; i++) {
                if (side == 0) in[i] = red[i];
                else in[M + i] = red[i];
            }
        }
        in[2 * M] = f1; in[2 * M + 1] = f2; in[2 * M + 2] = f3;
        float o0 = 0.0f, o1 = 0.0f, o2 = 0.0f;
#pragma unroll 1
        for (int j = 0; j < H; j += 4) {
            float h0 = 0.0f, h1 = 0.0f, h2 = 0.0f, h3 = 0.0f;
#pragma unroll
            for (int k = 0; k < 2 * M + 3; k++) {
                const float4 wv = w.ld4(Lay::W3 + k * H + j);
                h0 = FB_FMA(in[k], wv.x, h0);
                h1 = FB_FMA(in[k], wv.y, h1);
                h2 = FB_FMA(in[k], wv.z, h2);
                h3 = FB_FMA(in[k], wv.w, h3);
            }
            if (use_bias) {
                const float4 bb = w.ld4(Lay::b3 + j);
                h0 = FB_ADD(h0, bb.x); h1 = FB_ADD(h1, bb.y); h2 = FB_ADD(h2, bb.z); h3 = FB_ADD(h3, bb.w);
            }
            const float hh[4] = { gnn_act<MATH>(act, h0), gnn_act<MATH>(act, h1), gnn_act<MATH>(act, h2), gnn_act<MATH>(act, h3) };
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
                o0 = FB_FMA(hh[jj], w.ld(Lay::W0 + (j + jj) * 3 + 0), o0);
                o1 = FB_FMA(hh[jj], w.ld(Lay::W0 + (j + jj) * 3 + 1), o1);
                o2 = FB_FMA(hh[jj], w.ld(Lay::W0 + (j + jj) * 3 + 2), o2);
            }
        }
        if (use_bias) {
            o0 = FB_ADD(o0, w.ld(Lay::b0 + 0)); o1 = FB_ADD(o1, w.ld(Lay::b0 + 1)); o2 = FB_ADD(o2, w.ld(Lay::b0 + 2));
        }
        a.out(b, v, 0) = o0; a.out(b, v, 1) = o1; a.out(b, v, 2) = o2;
    }
}

// 96 registers, 5 CTAs / SM, with the regular path's hidden-unit loop not unrolled: measured best on B200
// (profiles/r02_lab_k_bp4_variants.txt, the k_gnn unroll / occupancy block: 319.5 k frames/s; unrolled by 2: 319.0 k;
// 4 CTAs / SM: 316.2 k; 6 CTAs / SM: 314.2 k)
template <int H, int M, int DV, bool TANH_BIAS, bool FACT, typename MATH>
static __global__ void __launch_bounds__(128, 5) k_gnn(const GnnArgs a) {
    extern __shared__ float wsm[];
    for (int i = threadIdx.x; i < GnnLayout<H, M>::total; i += blockDim.x) wsm[i] = a.weights[i];
    __syncthreads();
    gnn_body<H, M, DV, TANH_BIAS, FACT, MATH>(a, WSmem{wsm});
}

// ---- feedback GNN with MLPs of any depth (num_mlp_layers != 2; feedback_gnn.py:110-127) ----------------------------
// General form: every edge's MLP evaluated in full, messages reduced in edge order; arithmetic and packed weight layout
// are those of oracle/fbgnn_oracle.c (gnnd_vn).  One thread per (frame, variable node); the layer vectors live in local
// memory and the weights are read through the read-only cache -- this is the path for configurations outside the shipped
// one, not a tuned kernel.
constexpr int GNND_MAX = 128;

struct GnnDeepArgs {
    GnnArgs g;                          // graph tables, views, frame list (weights / act / reduce / use_bias of g are used)
    int H, M, L;
};

template <typename MATH>
__device__ __forceinline__ const float *gnnd_dense(const float *__restrict__ w, int kin, int kout, bool use_bias, int act,
                                                   const float *in, float *out) {
    for (int j = 0; j < kout; j++) {
        float a = 0.0f;
        for (int k = 0; k < kin; k++) a = FB_FMA(in[k], __ldg(w + k * kout + j), a);
        if (use_bias) a = FB_ADD(a, __ldg(w + kin * kout + j));
        out[j] = gnn_act<MATH>(act, a);
    }
    return w + kin * kout + kout;
}

template <typename MATH>
static __global__ void __launch_bounds__(128) k_gnn_deep(const GnnDeepArgs d) {
    const GnnArgs &a = d.g;
    const int n = a.X.n, H = d.H, M = d.M, L = d.L;
    const bool use_bias = a.use_bias != 0;
    const int64_t items = a.num_frames * n;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t fi = it / n;
        const int v = (int)(it - fi * n);
        const int64_t b = a.frame_list ? a.frame_list[fi] : fi;
        const float f3[3] = {a.h_vn(b, v, 0), a.h_vn(b, v, 1), a.h_vn(b, v, 2)};
        float in[2 * GNND_MAX + 3], va[GNND_MAX], vc[GNND_MAX];
        const float *w_inv = a.weights;
        const float *w = w_inv + ((L == 1 ? 2 * M + 3 : H) * 3 + 3);
        for (int side = 0; side < 2; side++) {
            const SideDev &S = side ? a.Z : a.X;
            const View2<const float> &logit = side ? a.logit_hz : a.logit_hx;
            const View2<const uint8_t> &synd = side ? a.sz : a.sx;
            float *red = in + side * M;
            const int e0 = S.vn_ptr[v], e1 = S.vn_ptr[v + 1];
            const float *wend = w;
            for (int i = 0; i < M; i++) red[i] = 0.0f;
            for (int e = e0; e < e1; e++) {
                const int c = S.vn_cn[e];
                va[0] = FB_MUL(logit(c, b), synd(c, b) ? -1.0f : 1.0f);
                va[1] = f3[0]; va[2] = f3[1]; va[3] = f3[2];
                const float *wl = w;
                int kin = 4;
                float *src = va, *dst = vc;
                for (int l = 0; l < L; l++) {
                    const int kout = (l == L - 1) ? M : H;
                    wl = gnnd_dense<MATH>(wl, kin, kout, use_bias, (l == L - 1) ? 2 : a.act, src, dst);
                    float *t = src; src = dst; dst = t;
                    kin = kout;
                }
                wend = wl;
                for (int i = 0; i < M; i++) {
                    if (e == e0) red[i] = src[i];
                    else if (a.reduce <= 1) red[i] = FB_ADD(red[i], src[i]);
                    else if (a.reduce == 2) red[i] = (src[i] > red[i]) ? src[i] : red[i];
                    else red[i] = (src[i] < red[i]) ? src[i] : red[i];
                }
            }
            if (e1 == e0) {
                int kin = 4;
                for (int l = 0; l < L; l++) { const int kout = (l == L - 1) ? M : H; wend += kin * kout + kout; kin = kout; }
            } else if (a.reduce == 0) {
                const float deg = (float)(e1 - e0);
                for (int i = 0; i < M; i++) red[i] = FB_DIV(red[i], deg);
            }
            w = wend;
        }
        in[2 * M] = f3[0]; in[2 * M + 1] = f3[1]; in[2 * M + 2] = f3[2];
        float *src = in, *dst = va;
        int kin = 2 * M + 3;
        for (int l = 0; l < L - 1; l++) {
            w = gnnd_dense<MATH>(w, kin, H, use_bias, a.act, src, dst);
            src = dst; dst = (dst == va) ? vc : va;
            kin = H;
        }
        float o[3];
        gnnd_dense<MATH>(w_inv, kin, 3, use_bias, 2, src, o);
        a.out(b, v, 0) = o[0]; a.out(b, v, 1) = o[1]; a.out(b, v, 2) = o[2];
    }
}

// ------------------------------------------------------------------ GNN_BP4 -----------
// The full GNN message-passing decoder of gnn.py:71-751 (BASELINE configs[4]); arithmetic and
// summation orders are those of oracle/fbgnn_oracle.c (gbp_*).  Embeddings live in HBM
// ([B][nodes][D] float); one thread owns one receiving node of one frame, walks its edges, runs the
// edge MLP (2D -> H -> M) per edge with the receiver half of the first layer hoisted out of the edge
// loop, reduces, and runs the node MLP.  Weights are staged in shared memory.
template <int D, int H, int M> struct GbpLayout {
    static constexpr __host__ __device__ int pad4(int x) { return (x + 3) & ~3; }
    static constexpr int edge = pad4(H * 2 * D) + pad4(H) + pad4(H * M) + pad4(M);        // W1T[H][2D], b1, W2[H][M], b2
    static constexpr int e_b1 = pad4(H * 2 * D), e_W2 = e_b1 + pad4(H), e_b2 = e_W2 + pad4(H * M);
    static constexpr __host__ __device__ int node(int K) { return pad4(K * H) + pad4(H) + pad4(H * D) + pad4(D); }   // W1[K][H], b1, W2[H][D], b2
    static constexpr __host__ __device__ int n_b1(int K) { return pad4(K * H); }
    static constexpr __host__ __device__ int n_W2(int K) { return pad4(K * H) + pad4(H); }
    static constexpr __host__ __device__ int n_b2(int K) { return pad4(K * H) + pad4(H) + pad4(H * D); }
    static constexpr int KC = M + D + 1, KV = 2 * M + D;
    // CN kernel: [edge x][edge z][node x][node z];  VN kernel: [edge x][edge z][node]
    static constexpr int cn_total = 2 * edge + 2 * node(KC);
    static constexpr int vn_total = 2 * edge + node(KV);
};

struct GbpArgs {
    SideDev X, Z;
    const float *w_cn, *w_vn;           // packed weights of update_h_cn / update_h_vn (GbpLayout)
    const float *w_inv;                 // [D][3] + [3] (bias, zeros if unused)
    int act, reduce, use_bias;
    int64_t B;
    float *h_vn, *hcx, *hcz;            // [B][n][D], [B][m_x][D], [B][m_z][D]
    float *lg;                          // [B][m_x + m_z]: hx_logit, hz_logit of the last cal_logit
    // factored form (reduce mean / sum): sender halves of the first edge layer, written by the kernel that
    // produces the sender's embedding and read once per edge by the receiving side
    float *pfc;                         // [B][m_x + m_z][H]: W1[:D]^T h_cn with update_h_vn's msg_mlp_{x,z}
    float *pfv;                         // [B][n][2][H]:      W1[:D]^T h_vn with update_h_cn's msg_mlp_{x,z}
    const uint8_t *sx, *sz;             // [B][m_x], [B][m_z] (batch first, gnn.py:385-386)
    int zero_logits;                    // first CN update: logits are zero
    // cal_logit outputs (optional) and logical rows
    const int *lx_ptr, *lz_ptr; const idx_t *lx_col, *lz_col; int kx, kz;
    View2<float> x_logit, z_logit;      // (row, b) slices of this iteration: [m_z + k_z], [m_x + k_x]
    View2<uint8_t> x_hat, z_hat;        // (v, b) optional (last iteration)
};

template <typename MATH>
__device__ __forceinline__ float gbp_act(int act, float x) { return gnn_act<MATH>(act, x); }

// msg = W2^T act(base + W1s^T from + b1) + b2, reduced into red[] (order: oracle gbp_edge_mlp / gbp_reduce)
template <int D, int H, int M, typename MATH>
__device__ __forceinline__ void gbp_edge(const float *__restrict__ w, const float *base_s, int bstride,
                                         const float from[D], int act, bool use_bias, bool negate, bool first,
                                         int reduce, float red[M]) {
    typedef GbpLayout<D, H, M> L;
    float acc[M];
#pragma unroll
    for (int i = 0; i < M; i++) acc[i] = 0.0f;
#pragma unroll 2
    for (int j = 0; j < H; j++) {
        float a = base_s[j * bstride];
        const float *w1 = w + j * 2 * D;
#pragma unroll
        for (int k = 0; k < D; k += 4) {
            const float4 wv = *reinterpret_cast<const float4 *>(w1 + k);
            a = FB_FMA(from[k + 0], wv.x, a); a = FB_FMA(from[k + 1], wv.y, a);
            a = FB_FMA(from[k + 2], wv.z, a); a = FB_FMA(from[k + 3], wv.w, a);
        }
        if (use_bias) a = FB_ADD(a, w[L::e_b1 + j]);
        const float hv = gbp_act<MATH>(act, a);
        const float *w2 = w + L::e_W2 + j * M;
#pragma unroll
        for (int i = 0; i < M; i += 4) {
            const float4 wv = *reinterpret_cast<const float4 *>(w2 + i);
            acc[i + 0] = FB_FMA(hv, wv.x, acc[i + 0]); acc[i + 1] = FB_FMA(hv, wv.y, acc[i + 1]);
            acc[i + 2] = FB_FMA(hv, wv.z, acc[i + 2]); acc[i + 3] = FB_FMA(hv, wv.w, acc[i + 3]);
        }
    }
#pragma unroll
    for (int i = 0; i < M; i++) {
        float mval = use_bias ? FB_ADD(acc[i], w[L::e_b2 + i]) : acc[i];
        if (negate) mval = -mval;
        if (first) red[i] = (reduce <= 1) ? FB_ADD(0.0f, mval) : mval;
        else if (reduce <= 1) red[i] = FB_ADD(red[i], mval);
        else if (reduce == 2) red[i] = (mval > red[i]) ? mval : red[i];
        else red[i] = (mval < red[i]) ? mval : red[i];
    }
}

// receiver half of the first edge layer: base[j] = sum_k to[k] * W1[D + k][j]
template <int D, int H, int M>
__device__ __forceinline__ void gbp_base(const float *__restrict__ w, const float to[D], float *base_s, int bstride) {
#pragma unroll 2
    for (int j = 0; j < H; j++) {
        float a = 0.0f;
        const float *w1 = w + j * 2 * D + D;
#pragma unroll
        for (int k = 0; k < D; k += 4) {
            const float4 wv = *reinterpret_cast<const float4 *>(w1 + k);
            a = FB_FMA(to[k + 0], wv.x, a); a = FB_FMA(to[k + 1], wv.y, a);
            a = FB_FMA(to[k + 2], wv.z, a); a = FB_FMA(to[k + 3], wv.w, a);
        }
        base_s[j * bstride] = a;
    }
}

// node MLP: out = W2^T act(W1^T in + b1) + b2 with in[K] in registers (order: oracle gbp_node_mlp)
template <int D, int H, int M, int K, typename MATH>
__device__ __forceinline__ void gbp_node(const float *__restrict__ w, const float in[K], int act, bool use_bias,
                                         float out[D]) {
    typedef GbpLayout<D, H, M> L;
#pragma unroll
    for (int i = 0; i < D; i++) out[i] = 0.0f;
#pragma unroll 1
    for (int j = 0; j < H; j += 4) {
        float h0 = 0.0f, h1 = 0.0f, h2 = 0.0f, h3 = 0.0f;
#pragma unroll
        for (int k = 0; k < K; k++) {
            const float4 wv = *reinterpret_cast<const float4 *>(w + k * H + j);
            h0 = FB_FMA(in[k], wv.x, h0); h1 = FB_FMA(in[k], wv.y, h1);
            h2 = FB_FMA(in[k], wv.z, h2); h3 = FB_FMA(in[k], wv.w, h3);
        }
        if (use_bias) {
            const float4 bb = *reinterpret_cast<const float4 *>(w + L::n_b1(K) + j);
            h0 = FB_ADD(h0, bb.x); h1 = FB_ADD(h1, bb.y); h2 = FB_ADD(h2, bb.z); h3 = FB_ADD(h3, bb.w);
        }
        const float hh[4] = { gbp_act<MATH>(act, h0), gbp_act<MATH>(act, h1), gbp_act<MATH>(act, h2), gbp_act<MATH>(act, h3) };
#pragma unroll
        for (int jj = 0; jj < 4; jj++) {
            const float *w2 = w + L::n_W2(K) + (j + jj) * D;
#pragma unroll
            for (int i = 0; i < D; i += 4) {
                const float4 wv = *reinterpret_cast<const float4 *>(w2 + i);
                out[i + 0] = FB_FMA(hh[jj], wv.x, out[i + 0]); out[i + 1] = FB_FMA(hh[jj], wv.y, out[i + 1]);
                out[i + 2] = FB_FMA(hh[jj], wv.z, out[i + 2]); out[i + 3] = FB_FMA(hh[jj], wv.w, out[i + 3]);
            }
        }
    }
    if (use_bias) {
#pragma unroll
        for (int i = 0; i < D; i++) out[i] = FB_ADD(out[i], w[L::n_b2(K) + i]);
    }
}

// UpdateCNEmbeddings.call (gnn.py:574-610): one thread per (frame, check), X checks then Z checks.
// smem: weights[cn_total] + base[H][blockDim]
template <int D, int H, int M, typename MATH>
static __global__ void __launch_bounds__(128) k_gbp_cn(const GbpArgs a) {
    typedef GbpLayout<D, H, M> L;
    extern __shared__ float gsm[];
    float *w = gsm, *base = gsm + L::cn_total + threadIdx.x;
    for (int i = threadIdx.x; i < L::cn_total; i += blockDim.x) w[i] = a.w_cn[i];
    __syncthreads();
    const int mt = a.X.m + a.Z.m;
    const bool use_bias = a.use_bias != 0;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < a.B * mt; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = it / mt;
        const int c = (int)(it - b * mt);
        const bool isx = c < a.X.m;
        const SideDev &S = isx ? a.X : a.Z;
        const int cc = isx ? c : c - a.X.m;
        const float *we = w + (isx ? 0 : L::edge), *wn = w + 2 * L::edge + (isx ? 0 : L::node(L::KC));
        float *hc = (isx ? a.hcx + (b * a.X.m + cc) * D : a.hcz + (b * a.Z.m + cc) * D);
        float in[L::KC], own[D];
#pragma unroll
        for (int k = 0; k < D; k += 4) {
            const float4 v4 = *reinterpret_cast<const float4 *>(hc + k);
            own[k] = v4.x; own[k + 1] = v4.y; own[k + 2] = v4.z; own[k + 3] = v4.w;
        }
        gbp_base<D, H, M>(we, own, base, blockDim.x);
        float red[M];
#pragma unroll
        for (int i = 0; i < M; i++) red[i] = 0.0f;
        const int k0 = S.cn_ptr[cc], k1 = S.cn_ptr[cc + 1];
        for (int k = k0; k < k1; k++) {
            const float *hv = a.h_vn + (b * S.n + S.cn_vn[k]) * D;
            float from[D];
#pragma unroll
            for (int q = 0; q < D; q += 4) {
                const float4 v4 = *reinterpret_cast<const float4 *>(hv + q);
                from[q] = v4.x; from[q + 1] = v4.y; from[q + 2] = v4.z; from[q + 3] = v4.w;
            }
            gbp_edge<D, H, M, MATH>(we, base, blockDim.x, from, a.act, use_bias, false, k == k0, a.reduce, red);
        }
        if (a.reduce == 0 && k1 > k0) {
            const float dg = (float)(k1 - k0);
#pragma unroll
            for (int i = 0; i < M; i++) red[i] = FB_DIV(red[i], dg);
        }
#pragma unroll
        for (int i = 0; i < M; i++) in[i] = red[i];
#pragma unroll
        for (int i = 0; i < D; i++) in[M + i] = own[i];
        float lgv = 0.0f;
        if (!a.zero_logits) {
            lgv = a.lg[b * mt + c];
            if ((isx ? a.sx[b * a.X.m + cc] : a.sz[b * a.Z.m + cc])) lgv = -lgv;      // logit * (1 - 2 s)
        }
        in[M + D] = lgv;
        float out[D];
        gbp_node<D, H, M, L::KC, MATH>(wn, in, a.act, use_bias, out);
#pragma unroll
        for (int k = 0; k < D; k += 4) *reinterpret_cast<float4 *>(hc + k) = make_float4(out[k], out[k + 1], out[k + 2], out[k + 3]);
    }
}

// UpdateVNEmbeddings.call (gnn.py:716-750): one thread per (frame, variable node)
template <int D, int H, int M, typename MATH>
static __global__ void __launch_bounds__(128) k_gbp_vn(const GbpArgs a) {
    typedef GbpLayout<D, H, M> L;
    extern __shared__ float gsm[];
    float *w = gsm, *base = gsm + L::vn_total + threadIdx.x;
    for (int i = threadIdx.x; i < L::vn_total; i += blockDim.x) w[i] = a.w_vn[i];
    __syncthreads();
    const int n = a.X.n;
    const bool use_bias = a.use_bias != 0;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < a.B * n; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = it / n;
        const int v = (int)(it - b * n);
        float *hv = a.h_vn + (b * n + v) * D;
        float in[L::KV], own[D];
#pragma unroll
        for (int k = 0; k < D; k += 4) {
            const float4 v4 = *reinterpret_cast<const float4 *>(hv + k);
            own[k] = v4.x; own[k + 1] = v4.y; own[k + 2] = v4.z; own[k + 3] = v4.w;
        }
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
            const SideDev &S = side ? a.Z : a.X;
            const float *we = w + (side ? L::edge : 0);
            const float *hc = side ? a.hcz + b * a.Z.m * D : a.hcx + b * a.X.m * D;
            const uint8_t *sy = side ? a.sz + b * a.Z.m : a.sx + b * a.X.m;
            gbp_base<D, H, M>(we, own, base, blockDim.x);
            float red[M];
#pragma unroll
            for (int i = 0; i < M; i++) red[i] = 0.0f;
            const int e0 = S.vn_ptr[v], e1 = S.vn_ptr[v + 1];
            for (int e = e0; e < e1; e++) {
                const int c = S.vn_cn[e];
                float from[D];
#pragma unroll
                for (int q = 0; q < D; q += 4) {
                    const float4 v4 = *reinterpret_cast<const float4 *>(hc + c * D + q);
                    from[q] = v4.x; from[q + 1] = v4.y; from[q + 2] = v4.z; from[q + 3] = v4.w;
                }
                gbp_edge<D, H, M, MATH>(we, base, blockDim.x, from, a.act, use_bias, sy[c] != 0, e == e0, a.reduce, red);
            }
            if (a.reduce == 0 && e1 > e0) {
                const float dg = (float)(e1 - e0);
#pragma unroll
                for (int i = 0; i < M; i++) red[i] = FB_DIV(red[i], dg);
            }
#pragma unroll
            for (int i = 0; i < M; i++) {
                if (side == 0) in[i] = red[i];
                else in[M + i] = red[i];
            }
        }
#pragma unroll
        for (int i = 0; i < D; i++) in[2 * M + i] = own[i];
        float out[D];
        gbp_node<D, H, M, L::KV, MATH>(w + 2 * L::edge, in, a.act, use_bias, out);
#pragma unroll
        for (int k = 0; k < D; k += 4) *reinterpret_cast<float4 *>(hv + k) = make_float4(out[k], out[k + 1], out[k + 2], out[k + 3]);
    }
}

// ---- factored form for reduce_op "mean" / "sum" (arithmetic: oracle gbp_from / gbp_hidden_acc / gbp_out_layer)
// The first edge layer is linear in [h_from, h_to]: its sender half Pf = W1[:D]^T h_from is formed ONCE per
// sender node (by the kernel that writes that node's embedding), its receiver half once per receiver, and an
// edge only adds the two.  The output layer is linear too and is applied once per receiver to the signed sum
// of hidden activations.  Per edge that leaves H additions and H activations instead of 2 H (D + M) FMAs.

// Pf[j] = sum_k h[k] W1T[j][k]  (k < D), written as H floats
template <int D, int H>
__device__ __forceinline__ void gbp_sender_half(const float *__restrict__ w1t, const float h[D], float *__restrict__ dst) {
#pragma unroll 1
    for (int j = 0; j < H; j += 4) {
        float p[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            float acc = 0.0f;
            const float *w1 = w1t + (j + q) * D;
#pragma unroll
            for (int k = 0; k < D; k += 4) {
                const float4 wv = *reinterpret_cast<const float4 *>(w1 + k);
                acc = FB_FMA(h[k + 0], wv.x, acc); acc = FB_FMA(h[k + 1], wv.y, acc);
                acc = FB_FMA(h[k + 2], wv.z, acc); acc = FB_FMA(h[k + 3], wv.w, acc);
            }
            p[q] = acc;
        }
        *reinterpret_cast<float4 *>(dst + j) = make_float4(p[0], p[1], p[2], p[3]);
    }
}

// Messages into one receiver over edges [e0, e1).  SENDER(e) gives the edge's code: (row number of the sender
// in `rows`, row_stride floats apart) << 1 | (1 if the message is negated).  red[M] receives the reduced
// message.  The codes of the first GBP_CODE_CAP edges are staged once in the thread's shared-memory slots
// (codes[k * cstride]) so the hidden-unit steps below do not repeat the dependent index / syndrome loads.
// Hidden units are walked eight at a time (one 32-byte sector of every sender row per step); the row of edge
// e+1 is requested before edge e is evaluated and the first row of the next step before the output-layer
// products of this one, without unrolling the edge loop (its body stays inside the instruction cache).
constexpr int GBP_CODE_CAP = 8;

template <typename SENDER>
__device__ __forceinline__ void gbp_stage_codes(uint32_t *codes, int cstride, int e0, int e1, SENDER sender) {
    const int ne = min(e1 - e0, GBP_CODE_CAP);
    for (int k = 0; k < ne; k++) codes[k * cstride] = sender(e0 + k);
}

template <int D, int H, int M, typename MATH, typename SENDER>
__device__ __forceinline__ void gbp_recv_factored(const float *__restrict__ w, const float own[D], int e0, int e1, int act,
                                                  bool use_bias, int reduce, const float *__restrict__ rows, int row_stride,
                                                  uint32_t *codes, int cstride, SENDER sender, float red[M]) {
    typedef GbpLayout<D, H, M> L;
    constexpr int JB = 8;
    static_assert(H % JB == 0, "H must be a multiple of 8");
    gbp_stage_codes(codes, cstride, e0, e1, sender);
    auto code_at = [&](int e) -> uint32_t { return (e - e0 < GBP_CODE_CAP) ? codes[(e - e0) * cstride] : sender(e); };
#pragma unroll
    for (int i = 0; i < M; i++) red[i] = 0.0f;
    int ssum = 0;
    uint32_t c0 = 0;
    float4 nx0 = make_float4(0.0f, 0.0f, 0.0f, 0.0f), nx1 = nx0;
    if (e0 < e1) {
        c0 = code_at(e0);
        const float *pf = rows + (int64_t)(c0 >> 1) * row_stride;
        nx0 = *reinterpret_cast<const float4 *>(pf); nx1 = *reinterpret_cast<const float4 *>(pf + 4);
    }
#pragma unroll 1
    for (int j = 0; j < H; j += JB) {
        float bs[JB], hs[JB], b1[JB];
#pragma unroll
        for (int q = 0; q < JB; q++) {          // receiver half of the first layer (oracle gbp_base)
            float acc = 0.0f;
            const float *w1 = w + (j + q) * 2 * D + D;
#pragma unroll
            for (int k = 0; k < D; k += 4) {
                const float4 wv = *reinterpret_cast<const float4 *>(w1 + k);
                acc = FB_FMA(own[k + 0], wv.x, acc); acc = FB_FMA(own[k + 1], wv.y, acc);
                acc = FB_FMA(own[k + 2], wv.z, acc); acc = FB_FMA(own[k + 3], wv.w, acc);
            }
            bs[q] = acc;
            hs[q] = 0.0f;
            b1[q] = use_bias ? w[L::e_b1 + j + q] : 0.0f;
        }
        uint32_t cc = c0;
#pragma unroll 1
        for (int e = e0; e < e1; e++) {
            const float pq[JB] = {nx0.x, nx0.y, nx0.z, nx0.w, nx1.x, nx1.y, nx1.z, nx1.w};
            const bool neg = (cc & 1u) != 0;
            if (e + 1 < e1) {
                cc = code_at(e + 1);
                const float *pf = rows + (int64_t)(cc >> 1) * row_stride + j;
                nx0 = *reinterpret_cast<const float4 *>(pf); nx1 = *reinterpret_cast<const float4 *>(pf + 4);
            }
            if (j == 0) ssum += neg ? -1 : 1;
#pragma unroll
            for (int q = 0; q < JB; q++) {
                float t = FB_ADD(pq[q], bs[q]);
                if (use_bias) t = FB_ADD(t, b1[q]);
                t = gbp_act<MATH>(act, t);
                if (neg) t = -t;
                hs[q] = (e == e0) ? t : FB_ADD(hs[q], t);
            }
        }
        if (j + JB < H && e0 < e1) {
            const float *pf = rows + (int64_t)(c0 >> 1) * row_stride + j + JB;
            nx0 = *reinterpret_cast<const float4 *>(pf); nx1 = *reinterpret_cast<const float4 *>(pf + 4);
        }
#pragma unroll
        for (int q = 0; q < JB; q++) {
            const float *w2 = w + L::e_W2 + (j + q) * M;
#pragma unroll
            for (int i = 0; i < M; i += 4) {
                const float4 wv = *reinterpret_cast<const float4 *>(w2 + i);
                red[i + 0] = FB_FMA(hs[q], wv.x, red[i + 0]); red[i + 1] = FB_FMA(hs[q], wv.y, red[i + 1]);
                red[i + 2] = FB_FMA(hs[q], wv.z, red[i + 2]); red[i + 3] = FB_FMA(hs[q], wv.w, red[i + 3]);
            }
        }
    }
    const float fs = (float)ssum, dg = (float)(e1 - e0);
#pragma unroll
    for (int i = 0; i < M; i++) {
        float r = red[i];
        if (use_bias) r = FB_FMA(fs, w[L::e_b2 + i], r);
        if (reduce == 0 && e1 > e0) r = FB_DIV(r, dg);
        red[i] = r;
    }
}

// initial sender halves of the variable nodes (h_vn as stored), before the first CN update
template <int D, int H, int M>
static __global__ void __launch_bounds__(128) k_gbp_pre_vn(const GbpArgs a) {
    typedef GbpLayout<D, H, M> L;
    extern __shared__ float gsm[];
    float *wp = gsm;                                                   // [2][H][D]
    for (int i = threadIdx.x; i < 2 * H * D; i += blockDim.x) {
        const int side = i / (H * D), r = i - side * H * D, j = r / D, k = r - j * D;
        wp[i] = a.w_cn[side * L::edge + j * 2 * D + k];
    }
    __syncthreads();
    const int n = a.X.n;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < a.B * n; it += (int64_t)gridDim.x * blockDim.x) {
        float own[D];
#pragma unroll
        for (int k = 0; k < D; k += 4) {
            const float4 v4 = *reinterpret_cast<const float4 *>(a.h_vn + it * D + k);
            own[k] = v4.x; own[k + 1] = v4.y; own[k + 2] = v4.z; own[k + 3] = v4.w;
        }
        gbp_sender_half<D, H>(wp, own, a.pfv + it * 2 * H);
        gbp_sender_half<D, H>(wp + H * D, own, a.pfv + it * 2 * H + H);
    }
}

// UpdateCNEmbeddings.call, factored; also writes the new check embedding's sender half for the VN update.
// smem: weights[cn_total] + sender-half weights of update_h_vn's msg_mlp_{x,z} [2][H][D]
template <int D, int H, int M, bool TB, typename MATH>
static __global__ void __launch_bounds__(128, 4) k_gbp_cn_f(const GbpArgs a) {
    typedef GbpLayout<D, H, M> L;
    extern __shared__ float gsm[];
    float *w = gsm, *wp = gsm + L::cn_total;
    uint32_t *codes = reinterpret_cast<uint32_t *>(wp + 2 * H * D) + threadIdx.x;      // [GBP_CODE_CAP][blockDim]
    for (int i = threadIdx.x; i < L::cn_total; i += blockDim.x) w[i] = a.w_cn[i];
    for (int i = threadIdx.x; i < 2 * H * D; i += blockDim.x) {
        const int side = i / (H * D), r = i - side * H * D, j = r / D, k = r - j * D;
        wp[i] = a.w_vn[side * L::edge + j * 2 * D + k];
    }
    __syncthreads();
    const int mt = a.X.m + a.Z.m, n = a.X.n;
    // TB: compile-time specialisation of tanh + use_bias=True (BASELINE configs[4]); keeps one copy of the loops
    const bool use_bias = TB ? true : (a.use_bias != 0);
    const int act = TB ? 0 : a.act;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < a.B * mt; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = it / mt;
        const int c = (int)(it - b * mt);
        const bool isx = c < a.X.m;
        const SideDev &S = isx ? a.X : a.Z;
        const int cc = isx ? c : c - a.X.m;
        const float *we = w + (isx ? 0 : L::edge), *wn = w + 2 * L::edge + (isx ? 0 : L::node(L::KC));
        float *hc = (isx ? a.hcx + (b * a.X.m + cc) * D : a.hcz + (b * a.Z.m + cc) * D);
        float in[L::KC], own[D];
#pragma unroll
        for (int k = 0; k < D; k += 4) {
            const float4 v4 = *reinterpret_cast<const float4 *>(hc + k);
            own[k] = v4.x; own[k + 1] = v4.y; own[k + 2] = v4.z; own[k + 3] = v4.w;
        }
        const float *pf_b = a.pfv + b * n * 2 * H + (isx ? 0 : H);
        const idx_t *cn_vn = S.cn_vn;
        float red[M];
        gbp_recv_factored<D, H, M, MATH>(we, own, S.cn_ptr[cc], S.cn_ptr[cc + 1], act, use_bias, a.reduce, pf_b, 2 * H,
            codes, blockDim.x, [&](int e) { return (uint32_t)cn_vn[e] << 1; }, red);
#pragma unroll
        for (int i = 0; i < M; i++) in[i] = red[i];
#pragma unroll
        for (int i = 0; i < D; i++) in[M + i] = own[i];
        float lgv = 0.0f;
        if (!a.zero_logits) {
            lgv = a.lg[b * mt + c];
            if ((isx ? a.sx[b * a.X.m + cc] : a.sz[b * a.Z.m + cc])) lgv = -lgv;      // logit * (1 - 2 s)
        }
        in[M + D] = lgv;
        float out[D];
        gbp_node<D, H, M, L::KC, MATH>(wn, in, act, use_bias, out);
#pragma unroll
        for (int k = 0; k < D; k += 4) *reinterpret_cast<float4 *>(hc + k) = make_float4(out[k], out[k + 1], out[k + 2], out[k + 3]);
        gbp_sender_half<D, H>(wp + (isx ? 0 : H * D), out, a.pfc + it * H);
    }
}

// UpdateVNEmbeddings.call, factored; also writes the new variable embedding's sender halves for the CN update.
template <int D, int H, int M, bool TB, typename MATH>
static __global__ void __launch_bounds__(128) k_gbp_vn_f(const GbpArgs a) {
    typedef GbpLayout<D, H, M> L;
    extern __shared__ float gsm[];
    float *w = gsm, *wp = gsm + L::vn_total;
    uint32_t *codes = reinterpret_cast<uint32_t *>(wp + 2 * H * D) + threadIdx.x;      // [GBP_CODE_CAP][blockDim]
    for (int i = threadIdx.x; i < L::vn_total; i += blockDim.x) w[i] = a.w_vn[i];
    for (int i = threadIdx.x; i < 2 * H * D; i += blockDim.x) {
        const int side = i / (H * D), r = i - side * H * D, j = r / D, k = r - j * D;
        wp[i] = a.w_cn[side * L::edge + j * 2 * D + k];
    }
    __syncthreads();
    const int n = a.X.n, mt = a.X.m + a.Z.m;
    // TB: compile-time specialisation of tanh + use_bias=True (BASELINE configs[4]); keeps one copy of the loops
    const bool use_bias = TB ? true : (a.use_bias != 0);
    const int act = TB ? 0 : a.act;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < a.B * n; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = it / n;
        const int v = (int)(it - b * n);
        float *hv = a.h_vn + it * D;
        float in[L::KV], own[D];
#pragma unroll
        for (int k = 0; k < D; k += 4) {
            const float4 v4 = *reinterpret_cast<const float4 *>(hv + k);
            own[k] = v4.x; own[k + 1] = v4.y; own[k + 2] = v4.z; own[k + 3] = v4.w;
        }
#pragma unroll 1
        for (int side = 0; side < 2; side++) {
            const SideDev &S = side ? a.Z : a.X;
            const float *pf_b = a.pfc + (b * mt + (side ? a.X.m : 0)) * H;
            const uint8_t *sy = side ? a.sz + b * a.Z.m : a.sx + b * a.X.m;
            const idx_t *vn_cn = S.vn_cn;
            float red[M];
            gbp_recv_factored<D, H, M, MATH>(w + (side ? L::edge : 0), own, S.vn_ptr[v], S.vn_ptr[v + 1], act, use_bias,
                a.reduce, pf_b, H, codes, blockDim.x,
                [&](int e) { const uint32_t c = vn_cn[e]; return (c << 1) | (sy[c] != 0 ? 1u : 0u); }, red);
#pragma unroll
            for (int i = 0; i < M; i++) {
                if (side == 0) in[i] = red[i];
                else in[M + i] = red[i];
            }
        }
#pragma unroll
        for (int i = 0; i < D; i++) in[2 * M + i] = own[i];
        float out[D];
        gbp_node<D, H, M, L::KV, MATH>(w + 2 * L::edge, in, act, use_bias, out);
#pragma unroll
        for (int k = 0; k < D; k += 4) *reinterpret_cast<float4 *>(hv + k) = make_float4(out[k], out[k + 1], out[k + 2], out[k + 3]);
        gbp_sender_half<D, H>(wp, out, a.pfv + it * 2 * H);
        gbp_sender_half<D, H>(wp + H * D, out, a.pfv + it * 2 * H + H);
    }
}

// embed_to_llr + cal_logit + make_hard_decision (gnn.py:281-314, 358-366): one CTA per frame.
// smem: float lxp[n], lzp[n] (phi2 of |llr_x'|, |llr_z'|); u8 sgn[n]
template <int D, typename MATH>
static __global__ void k_gbp_logit(const GbpArgs a) {
    extern __shared__ float lsm[];
    const int n = a.X.n, T = blockDim.x, tid = threadIdx.x;
    const int64_t b = blockIdx.x;
    float *px = lsm, *pz = px + n;
    uint8_t *sgn = (uint8_t *)(pz + n);
    for (int v = tid; v < n; v += T) {
        const float *hv = a.h_vn + (b * n + v) * D;
        float l[3];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            float acc = 0.0f;
#pragma unroll
            for (int k = 0; k < D; k++) acc = FB_FMA(hv[k], a.w_inv[k * 3 + c], acc);
            if (a.use_bias) acc = FB_ADD(acc, a.w_inv[D * 3 + c]);
            l[c] = acc;
        }
        const float lx = l[0], ly = l[1], lz = l[2];
        const float llr_zp = FB_SUB(MATH::softplus(-lx), MATH::logaddexp(-lz, -ly));
        const float llr_xp = FB_SUB(MATH::softplus(-lz), MATH::logaddexp(-lx, -ly));
        sgn[v] = (uint8_t)(((llr_xp < 0.0f) ? 1 : 0) | ((llr_zp < 0.0f) ? 2 : 0));
        px[v] = MATH::phi2(fabsf(llr_xp));
        pz[v] = MATH::phi2(fabsf(llr_zp));
        if (a.x_hat.ptr) {
            int d = 0;
            float best = 0.0f;
            if (lx < best) { best = lx; d = 1; }
            if (lz < best) { best = lz; d = 2; }
            if (ly < best) { best = ly; d = 3; }
            a.x_hat(v, b) = (uint8_t)(d & 1);
            a.z_hat(v, b) = (uint8_t)(d >> 1);
        }
    }
    __syncthreads();
    const int mx = a.X.m, mz = a.Z.m, total = mx + mz + a.kx + a.kz;
    for (int r = tid; r < total; r += T) {
        // rows: [hx (mx)] [hz (mz)] [lx (kx)] [lz (kz)];  hx / lx rows use llr_z', hz / lz rows use llr_x'
        const bool usez = r < mx || (r >= mx + mz && r < mx + mz + a.kx);
        const float *sc = usez ? pz : px;
        const int bit = usez ? 1 : 0;
        int par = 0;
        float Tsum = 0.0f;
        if (r < mx + mz) {
            const SideDev &S = r < mx ? a.X : a.Z;
            const int cc = r < mx ? r : r - mx;
            for (int k = S.cn_ptr[cc]; k < S.cn_ptr[cc + 1]; k++) {
                const int v = S.cn_vn[k];
                par ^= (sgn[v] >> bit) & 1;
                Tsum = FB_ADD(Tsum, sc[v]);
            }
        } else {
            const bool islx = r < mx + mz + a.kx;
            const int rr = islx ? r - mx - mz : r - mx - mz - a.kx;
            const int *ptr = islx ? a.lx_ptr : a.lz_ptr;
            const idx_t *col = islx ? a.lx_col : a.lz_col;
            for (int k = ptr[rr]; k < ptr[rr + 1]; k++) {
                const int v = col[k];
                par ^= (sgn[v] >> bit) & 1;
                Tsum = FB_ADD(Tsum, sc[v]);
            }
        }
        float val = MATH::phi2(Tsum);
        val = par ? -val : val;
        if (r < mx + mz) a.lg[b * (mx + mz) + r] = val;
        // x_perp_logit = [hz_logit; lz_logit], z_perp_logit = [hx_logit; lx_logit] (gnn.py:311-313)
        if (a.x_logit.ptr) {
            if (r >= mx && r < mx + mz) a.x_logit(r - mx, b) = val;
            else if (r >= mx + mz + a.kx) a.x_logit(mz + (r - mx - mz - a.kx), b) = val;
        }
        if (a.z_logit.ptr) {
            if (r < mx) a.z_logit(r, b) = val;
            else if (r >= mx + mz && r < mx + mz + a.kx) a.z_logit(mx + (r - mx - mz), b) = val;
        }
    }
}

// ------------------------------------------------------------------ noise + syndrome --
struct SampleArgs {
    SideDev X, Z;                       // Z.n == 0 for the binary (single pcm) pipeline
    int mode;                           // 0 Pauli depolarising, 1 BSC, 2 Pauli of fixed weight `wt` (pauli.py:80-96)
    int wt;
    float thr0, thr1, thr2;             // Pauli thresholds, or thr0 = p for BSC
    uint64_t seed, first_frame;
    View2<const uint8_t> nx_in, nz_in;  // optional given noise (b, v)
    const uint32_t *nx_words, *nz_words;   // optional given noise as packed bit-planes [B][wq]: qubit v = bit (v & 31) of word v >> 5
    int wq;                             // row stride of the packed planes in words
    uint8_t *vbits;                     // [B][n] out: bit0 noise_x (or BSC noise), bit1 noise_z
    uint8_t *sbits;                     // [B][sb_stride] out (may be nullptr): syndrome_x then syndrome_z of the frame
    int sb_stride;                      // row stride in bytes (pad16(m_x + m_z) in the pipelines' workspace)
    View2<uint8_t> nx_out, nz_out;      // optional separate outputs (Pauli / BSC layer API)
};

__device__ __forceinline__ float frame_uniform(uint64_t seed, uint64_t frame, uint32_t q, uint32_t stream) {
    uint32_t r[4];
    philox4x32_10((uint32_t)frame, (uint32_t)(frame >> 32), q >> 2, stream, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    return u01(r[q & 3]);
}

// smem: u8 nb[n] (+ u16 idx[n] in fixed-weight mode)
static __global__ void k_sample(const SampleArgs a) {
    extern __shared__ uint8_t nb[];
    const int n = a.X.n, T = blockDim.x, tid = threadIdx.x;
    const int64_t b = blockIdx.x;
    const uint64_t frame = a.first_frame + (uint64_t)b;
    if (a.nx_words) {                   // packed planes: coalesced 32-bit loads, 32 qubits per word
        const uint32_t *wx = a.nx_words + b * a.wq, *wz = a.nz_words ? a.nz_words + b * a.wq : nullptr;
        for (int v = tid; v < n; v += T)
            nb[v] = (uint8_t)(((wx[v >> 5] >> (v & 31)) & 1u) | (wz ? (((wz[v >> 5] >> (v & 31)) & 1u) << 1) : 0u));
    } else if (a.nx_in.ptr) {
        for (int v = tid; v < n; v += T)
            nb[v] = (a.nx_in(b, v) ? 1 : 0) | ((a.nz_in.ptr && a.nz_in(b, v)) ? 2 : 0);
    } else if (a.mode == 2) {
        // partial Fisher-Yates: the first wt entries of a shuffle, then the Pauli type of each position
        uint16_t *idx = (uint16_t *)(nb + ((n + 1) & ~1));
        for (int v = tid; v < n; v += T) { idx[v] = (uint16_t)v; nb[v] = 0; }
        __syncthreads();
        if (tid == 0) {
            const int wt = a.wt < n ? a.wt : n;
            for (int i = 0; i < wt; i++) {
                const float u = frame_uniform(a.seed, frame, (uint32_t)i, 2u);
                const int j = i + (int)FB_MUL(u, (float)(n - i));
                const uint16_t t = idx[i]; idx[i] = idx[j]; idx[j] = t;
                const float w = frame_uniform(a.seed, frame, (uint32_t)i, 3u);
                nb[idx[i]] = (uint8_t)((w < 0.6666667f ? 1 : 0) | (w > 0.33333334f ? 2 : 0));
            }
        }
    } else {
        for (int q4 = tid; q4 < (n + 3) / 4; q4 += T) {
            uint32_t r[4];
            philox4x32_10((uint32_t)frame, (uint32_t)(frame >> 32), (uint32_t)q4, (uint32_t)a.mode,
                          (uint32_t)a.seed, (uint32_t)(a.seed >> 32), r);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int q = q4 * 4 + j;
                if (q < n) {
                    const float u = u01(r[j]);
                    int bits;
                    if (a.mode != 1) bits = (u < a.thr0 ? 1 : 0) | ((u >= a.thr1 && u < a.thr2) ? 2 : 0);
                    else bits = (u < a.thr0) ? 1 : 0;
                    nb[q] = (uint8_t)bits;
                }
            }
        }
    }
    __syncthreads();
    if (a.vbits) for (int v = tid; v < n; v += T) a.vbits[b * n + v] = nb[v];
    if (a.nx_out.ptr) for (int v = tid; v < n; v += T) a.nx_out(b, v) = nb[v] & 1;
    if (a.nz_out.ptr) for (int v = tid; v < n; v += T) a.nz_out(b, v) = (nb[v] >> 1) & 1;
    if (a.sbits) {
        uint8_t *sb = a.sbits + b * a.sb_stride;
        for (int c = tid; c < a.X.m + a.Z.m; c += T) {
            const bool isx = c < a.X.m;                  // syndrome_x = hx . noise_z (bit1);
            const SideDev &S = isx ? a.X : a.Z;          // syndrome_z = hz . noise_x (bit0)
            const int cc = isx ? c : c - a.X.m;
            const int bit = (isx && a.mode != 1) ? 1 : 0;
            int par = 0;
            for (int k = S.cn_ptr[cc]; k < S.cn_ptr[cc + 1]; k++) par ^= (nb[S.cn_vn[k]] >> bit) & 1;
            sb[c] = (uint8_t)par;
        }
    }
}

struct SyndromeArgs {
    SideDev S;
    View2<const uint8_t> noise;         // (b, v)
    View2<uint8_t> synd;                // (c, b)
};
static __global__ void k_syndrome(const SyndromeArgs a) {
    extern __shared__ uint8_t nb[];
    const int64_t b = blockIdx.x;
    for (int v = threadIdx.x; v < a.S.n; v += blockDim.x) nb[v] = a.noise(b, v) & 1;
    __syncthreads();
    for (int c = threadIdx.x; c < a.S.m; c += blockDim.x) {
        int par = 0;
        for (int k = a.S.cn_ptr[c]; k < a.S.cn_ptr[c + 1]; k++) par ^= nb[a.S.cn_vn[k]];
        a.synd(c, b) = (uint8_t)par;
    }
}

// ------------------------------------------------------------------ OSD ---------------
// OSD0_Decoder (bp_osd.py:8-77) for the frames BP left with a syndrome mismatch: order the columns
// by increasing reliability (stable), then for every row of the full-rank basis take the first
// remaining one as pivot and eliminate it from all other rows of [H_perm | s]; the OSD-0 solution
// sits on the pivot columns.  One CTA per frame; the permuted bit matrix lives in shared memory, stored
// word-major (M[w * Rp + row]) so that the row-parallel XOR sweeps are conflict-free and the pivot
// row is a broadcast.
// With order lam > 0 the combination sweep (OSD-CS, Roffe et al. 2020) runs on that reduced matrix
// before it is discarded.  Over the non-pivot columns c_0 < c_1 < ... (least reliable first) the
// candidates T are, by index: 0 the empty set (OSD-0), 1 + i the single {c_i}, then the pairs
// {c_i, c_j}, i < j < min(lam, n - R), in lexicographic order.  T's solution is 1 on T and
// s'_r ^ XOR_{c in T} M[r, c] on pivot piv[r]; the candidate of least (Hamming weight, index) wins.
struct OsdArgs {
    SideDev S;                          // graph of the basis matrix: rows = the rank basis rows
    const int *frame_list;              // optional: CTA i handles frame frame_list[i]
    View2<const float> llr;             // (b, v) reliabilities; the sort key is sign * llr
    float sign;                         // +1, or -1 to sort by -llr (binary decoder's logits)
    View2<const uint8_t> synd;          // (row, b): reduced syndrome, or the full one with synd_row
    const idx_t *synd_row;              // optional [rank]: row of the full syndrome behind basis row r
    View2<uint8_t> e_hat;               // (b, v) optional output
    uint8_t *vbits;                     // optional [B][n]: the solution goes to bit `vbit` (pipeline mode)
    int vbit;
    int order;                          // 0: OSD-0; lam > 0: OSD-CS of order lam
    int npad;                           // power of two >= n
    int cv_off;                         // byte offset of the OSD-CS bit vectors in shared memory (order > 0)
};

__device__ __forceinline__ unsigned long long osd_key(float x, int idx) {
    uint32_t u = (uint32_t)__float_as_int(x);
    u ^= (u >> 31) ? 0xFFFFFFFFu : 0x80000000u;             // order-preserving map float -> uint
    return ((unsigned long long)u << 32) | (uint32_t)idx;
}

// pair q (lexicographic over i < j < lp) -> (i, j); row i of the triangle starts at i (2 lp - i - 1) / 2
__device__ __forceinline__ void osd_pair(int64_t q, int lp, int &i, int &j) {
    const double t = 2.0 * lp - 1.0;
    i = (int)((t - sqrt(t * t - 8.0 * (double)q)) * 0.5);
    i = max(0, min(i, lp - 2));
    auto start = [lp](int r) { return (int64_t)r * (2 * lp - r - 1) / 2; };
    while (i > 0 && start(i) > q) i--;
    while (i < lp - 2 && start(i + 1) <= q) i++;
    j = (int)(i + 1 + (q - start(i)));
}

// one warp: the first column < n set in row `row` of the word-major bit matrix M (row stride Rp), 0 if none; the same
// value in every lane.  wn = n / 32; last_mask keeps the columns < n of word wn.
__device__ __forceinline__ int osd_pivot(const uint32_t *M, int Rp, int row, int W, int wn, uint32_t last_mask, int lane) {
    int p = 0, found = 0;
    for (int w0 = 0; w0 < W && !found; w0 += 32) {
        const int w = w0 + lane;
        uint32_t word = w < W ? M[w * Rp + row] : 0u;
        if (w == wn) word &= last_mask;
        if (w > wn) word = 0u;
        const uint32_t vote = __ballot_sync(0xffffffffu, word != 0u);
        if (vote) {
            const int l = __ffs(vote) - 1;
            const uint32_t wsel = __shfl_sync(0xffffffffu, word, l);
            p = (w0 + l) * 32 + (__ffs(wsel) - 1);
            found = 1;
        }
    }
    return p;
}

// OSD-CS step 4c, for every thread of the CTA: fold the pairs of the first lp non-pivot columns (bit vectors cv[lp][RW]
// and s' in sv[RW]) into this thread's least (weight << 32 | index), then take the CTA's least into *best (set to ~0
// beforehand and read after a __syncthreads).  N is the number of non-pivot columns.
__device__ __forceinline__ void osd_cs_best(unsigned long long mine, const uint32_t *cv, const uint32_t *sv, int RW, int lp,
                                            int N, unsigned long long *best) {
    const int64_t P = (int64_t)lp * (lp - 1) / 2;
    for (int64_t q = threadIdx.x; q < P; q += blockDim.x) {
        int i, j;
        osd_pair(q, lp, i, j);
        int w = 2;
        for (int k = 0; k < RW; k++) w += __popc(sv[k] ^ cv[i * RW + k] ^ cv[j * RW + k]);
        mine = min(mine, ((unsigned long long)w << 32) | (uint32_t)(1 + N + q));
    }
    for (int o = 16; o > 0; o >>= 1) mine = min(mine, __shfl_xor_sync(0xffffffffu, mine, o));
    if ((threadIdx.x & 31) == 0) atomicMin(best, mine);
}

// candidate index -> its columns t0 / t1 (-1: none); np lists the non-pivot columns in increasing position
__device__ __forceinline__ void osd_cs_columns(uint32_t idx, int N, int lp, const uint16_t *np, int &t0, int &t1) {
    if (idx >= 1 && idx <= (uint32_t)N) t0 = np[idx - 1];
    else if (idx > (uint32_t)N) {
        int i, j;
        osd_pair((int64_t)idx - 1 - N, lp, i, j);
        t0 = np[i]; t1 = np[j];
    }
}

// Steps of k_osd that the cluster form (k_osd_cluster, fbgnn_osd_cluster.cuh) runs too.  Each is called by every thread
// of the CTA and ends with the CTA's writes visible to all its threads.

// 1. stable ascending sort of sign * llr(b, .) (bitonic network on (key, index) pairs): order[j] = the column at
//    position j, inv[v] = the position of column v
__device__ __forceinline__ void osd_sort(const OsdArgs &a, int64_t b, unsigned long long *keys, uint16_t *order,
                                         uint16_t *inv) {
    const int n = a.S.n, T = blockDim.x, tid = threadIdx.x;
    for (int i = tid; i < a.npad; i += T)
        keys[i] = i < n ? osd_key(a.sign * a.llr(b, i), i) : ~0ull;
    __syncthreads();
    for (int k = 2; k <= a.npad; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < a.npad; i += T) {
                const int l = i ^ j;
                if (l > i) {
                    const unsigned long long x = keys[i], y = keys[l];
                    const bool up = (i & k) == 0;
                    if ((x > y) == up) { keys[i] = y; keys[l] = x; }
                }
            }
            __syncthreads();
        }
    }
    for (int j = tid; j < n; j += T) {
        const int v = (int)(keys[j] & 0xFFFFFFFFull);
        order[j] = (uint16_t)v;
        inv[v] = (uint16_t)j;
    }
    __syncthreads();
}

// 2. basis rows r0 .. r0 + nr - 1 of the permuted [H | s] as rows 0 .. nr - 1 of the bit matrix M (word-major, row
//    stride Rp, W words), one thread per row
__device__ __forceinline__ void osd_build_rows(const OsdArgs &a, int64_t b, uint32_t *M, int Rp, const uint16_t *inv,
                                               int r0, int nr) {
    const SideDev &S = a.S;
    const int n = S.n, W = (n + 1 + 31) / 32, T = blockDim.x, tid = threadIdx.x;
    for (int i = tid; i < W * Rp; i += T) M[i] = 0u;
    __syncthreads();
    for (int i = tid; i < nr; i += T) {
        const int r = r0 + i;
        for (int k = S.cn_ptr[r]; k < S.cn_ptr[r + 1]; k++) {
            const int j = inv[S.cn_vn[k]];
            M[(j >> 5) * Rp + i] ^= 1u << (j & 31);
        }
        const int sr = a.synd_row ? a.synd_row[r] : r;
        if (a.synd(sr, b)) M[(n >> 5) * Rp + i] ^= 1u << (n & 31);
    }
    __syncthreads();
}

// 4a. the non-pivot columns in increasing position into np[0 .. *num - 1]; np (n entries) is overwritten
__device__ __forceinline__ void osd_cs_list(uint16_t *np, const uint16_t *piv, int n, int R, int *num) {
    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31;
    for (int j = tid; j < n; j += T) np[j] = 1;
    __syncthreads();
    for (int r = tid; r < R; r += T) np[piv[r]] = 0;
    __syncthreads();
    if (tid < 32) {
        int cnt = 0;
        for (int j0 = 0; j0 < n; j0 += 32) {                       // list position <= column: reads stay ahead of writes
            const int j = j0 + lane;
            const bool np_col = j < n && np[j];
            const uint32_t vote = __ballot_sync(0xffffffffu, np_col);
            if (np_col) np[cnt + __popc(vote & ((1u << lane) - 1u))] = (uint16_t)j;
            cnt += __popc(vote);
        }
        if (lane == 0) *num = cnt;
    }
    __syncthreads();
}

// 5. the solution on the pivot columns of bit-matrix rows 0 .. nr - 1 (their pivots in piv[0 .. nr - 1]) and, with
//    with_t, on the columns t0 / t1 of the winning candidate, mapped back through the permutation.  The frame's
//    outputs must have been cleared before.
__device__ __forceinline__ void osd_write_solution(const OsdArgs &a, int64_t b, const uint32_t *M, int Rp,
                                                   const uint16_t *order, const uint16_t *piv, int nr, int t0, int t1,
                                                   bool with_t) {
    const int n = a.S.n, wn = n >> 5, T = blockDim.x, tid = threadIdx.x;
    for (int r = tid; r < nr; r += T) {
        int sol = (M[wn * Rp + r] >> (n & 31)) & 1u;
        if (t0 >= 0) sol ^= (M[(t0 >> 5) * Rp + r] >> (t0 & 31)) & 1u;
        if (t1 >= 0) sol ^= (M[(t1 >> 5) * Rp + r] >> (t1 & 31)) & 1u;
        const int v = order[piv[r]];
        if (sol) {
            if (a.e_hat.ptr) a.e_hat(b, v) = 1;
            if (a.vbits) a.vbits[b * n + v] |= (uint8_t)(1u << a.vbit);
        }
    }
    if (with_t && tid == 0) {
        for (int e = 0; e < 2; e++) {
            const int c = e ? t1 : t0;
            if (c < 0) continue;
            const int v = order[c];
            if (a.e_hat.ptr) a.e_hat(b, v) = 1;
            if (a.vbits) a.vbits[b * n + v] |= (uint8_t)(1u << a.vbit);
        }
    }
}

// smem: max(npad * 8, W * Rp * 4) bytes shared by the sort keys and the matrix; u16 order[n], inv[n], piv[R];
// with order > 0, at cv_off: u32 cv[lp][RW] (the first lp non-pivot columns over the rows) and sv[RW] (s')
static __global__ void __launch_bounds__(256) k_osd(const OsdArgs a) {
    extern __shared__ unsigned long long osd_smem[];
    const SideDev &S = a.S;
    const int n = S.n, R = S.m, T = blockDim.x, tid = threadIdx.x;
    const int W = (n + 1 + 31) / 32, Rp = R | 1;                 // odd stride: no bank conflicts across words
    const int64_t b = a.frame_list ? a.frame_list[blockIdx.x] : blockIdx.x;
    unsigned long long *keys = osd_smem;
    uint32_t *M = (uint32_t *)osd_smem;
    const size_t main_bytes = ((size_t)a.npad * 8 > (size_t)W * Rp * 4) ? (size_t)a.npad * 8 : (size_t)W * Rp * 4;
    uint16_t *order = (uint16_t *)((uint8_t *)osd_smem + ((main_bytes + 7) & ~(size_t)7));
    uint16_t *inv = order + n, *piv = inv + n;
    __shared__ int cur_p;

    // 1. stable ascending sort of the reliabilities
    osd_sort(a, b, keys, order, inv);

    // 2. permuted [H | s] as a bit matrix, one thread per row
    osd_build_rows(a, b, M, Rp, inv, 0, R);

    // 3. row-wise elimination
    const int wn = n >> 5;
    const uint32_t last_mask = (n & 31) ? ((1u << (n & 31)) - 1u) : 0u;   // columns < n inside word wn
    for (int r = 0; r < R; r++) {
        if (tid < 32) {
            const int p = osd_pivot(M, Rp, r, W, wn, last_mask, tid);
            if (tid == 0) { cur_p = p; piv[r] = (uint16_t)p; }
        }
        __syncthreads();
        const int p = cur_p, pw = p >> 5;
        const uint32_t pm = 1u << (p & 31);
        for (int i = tid; i < R; i += T) {
            if (i != r && (M[pw * Rp + i] & pm)) {
                for (int w = pw; w < W; w++) M[w * Rp + i] ^= M[w * Rp + r];   // the pivot row is zero before word pw
            }
        }
        __syncthreads();
    }

    // 4. OSD-CS: the candidate of least (weight, index); t0 / t1 are its columns (-1: none)
    int t0 = -1, t1 = -1;
    if (a.order > 0) {
        __shared__ unsigned long long best;
        __shared__ int num_np;
        const int RW = (R + 31) / 32, lp = min(a.order, max(n - R, 0));
        const int lane = tid & 31, warp = tid >> 5, nw = T >> 5;
        uint32_t *cv = (uint32_t *)((uint8_t *)osd_smem + a.cv_off), *sv = cv + (size_t)lp * RW;
        // 4a. the non-pivot columns listed in inv (free since step 2); s' as a bit vector
        if (tid == 0) best = ~0ull;
        osd_cs_list(inv, piv, n, R, &num_np);
        for (int k = warp; k < RW; k += nw) {
            const int r = k * 32 + lane;
            const uint32_t v = __ballot_sync(0xffffffffu, r < R && ((M[wn * Rp + r] >> (n & 31)) & 1u));
            if (lane == 0) sv[k] = v;
        }
        __syncthreads();
        const int N = num_np;
        unsigned long long mine = ~0ull;
        if (tid == 0) {                                            // the empty set: OSD-0
            int w = 0;
            for (int k = 0; k < RW; k++) w += __popc(sv[k]);
            mine = (unsigned long long)w << 32;
        }
        // 4b. single columns: a warp ballots 32 rows at a time (conflict-free) and keeps the first lp as bit vectors
        for (int i = warp; i < N; i += nw) {
            const int c = inv[i], cw = c >> 5;
            const uint32_t cm = 1u << (c & 31);
            int w = 1;
            for (int k = 0; k < RW; k++) {
                const int r = k * 32 + lane;
                const uint32_t v = __ballot_sync(0xffffffffu, r < R && (M[cw * Rp + r] & cm));
                if (i < lp && lane == 0) cv[i * RW + k] = v;
                w += __popc(v ^ sv[k]);
            }
            if (lane == 0) mine = min(mine, ((unsigned long long)w << 32) | (uint32_t)(1 + i));
        }
        __syncthreads();
        // 4c. pairs of the first lp columns, one thread per pair
        osd_cs_best(mine, cv, sv, RW, lp, N, &best);
        __syncthreads();
        osd_cs_columns((uint32_t)best, N, lp, inv, t0, t1);
    }

    // 5. the solution on the pivot columns and on T, mapped back through the permutation
    if (a.e_hat.ptr) for (int v = tid; v < n; v += T) a.e_hat(b, v) = 0;
    if (a.vbits) for (int v = tid; v < n; v += T) a.vbits[b * n + v] &= (uint8_t)~(1u << a.vbit);
    __syncthreads();
    osd_write_solution(a, b, M, Rp, order, piv, R, t0, t1, true);
}

// reliabilities handed to OSD-0 by BP4_OSD_Model (bp_osd.py:135-144), for the listed frames:
// out plane 0 = osd_llrx = softplus(-Lz) - logsumexp(-Lx, -Ly), plane 1 = osd_llrz (x <-> z)
struct OsdLlrArgs {
    int n;
    const int *frame_list;
    int64_t num_frames;
    const float *L;                     // [B][3][n]
    float *out;                         // [B][3][np] (planes 0, 1 written)
    int np;                             // plane stride of out (pad4(n) in the pipelines' workspace)
};
template <typename MATH>
static __global__ void k_osd_llr(const OsdLlrArgs a) {
    const int64_t items = a.num_frames * a.n;
    for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
        const int64_t fi = it / a.n;
        const int v = (int)(it - fi * a.n);
        const int64_t b = a.frame_list ? a.frame_list[fi] : fi;
        const float *L = a.L + b * 3 * a.n;
        const float lx = L[v], ly = L[a.n + v], lz = L[2 * a.n + v];
        a.out[b * 3 * a.np + a.np + v] = FB_SUB(MATH::softplus(-lx), MATH::logaddexp(-lz, -ly));
        a.out[b * 3 * a.np + v] = FB_SUB(MATH::softplus(-lz), MATH::logaddexp(-lx, -ly));
    }
}

// ------------------------------------------------------------------ final checks ------
struct FinalArgs {
    SideDev X, Z;                       // binary pipeline: X = pcm, Z.n == 0
    const uint32_t *lx_bits, *lz_bits;  // [k][W] logical operators (binary: lx_bits = logical pcm rows)
    int kx, kz;
    int binary;
    const uint8_t *vbits;               // [B][n]  (binary: bit0 noise, bit2 hard decision)
    const uint8_t *rounds;              // [B] or nullptr
    uint8_t *flags;                     // [B] or nullptr
    View2<uint8_t> x_diff, z_diff;      // optional (b, v)
    unsigned long long *counters;       // [4] device: frames, flagged, block, stage-0 failures
    // packed outputs (optional): per-frame indicator planes [3][fw] (flagged, block error, failed stage 0; frame b = bit b & 31
    // of word b >> 5; cleared by the caller) and the residual errors as bit-planes [B][wq]
    uint32_t *frame_bits;
    int64_t fw;
    uint32_t *xd_words, *zd_words;
    int wq;
};

// smem: u8 d[n]; u32 xw[W], zw[W]
static __global__ void k_final(const FinalArgs a) {
    extern __shared__ uint8_t dsm[];
    const int n = a.X.n, T = blockDim.x, tid = threadIdx.x, W = (n + 31) / 32;
    const int64_t b = blockIdx.x;
    uint8_t *d = dsm;
    uint32_t *xw = (uint32_t *)(dsm + ((n + 3) & ~3)), *zw = xw + W;
    // residual error after correction (feedback_gnn.py:346-347): bit0 x_diff, bit1 z_diff
    const int nround = ((n + 31) / 32) * 32;
    for (int v = tid; v < nround; v += T) {
        int bits = 0;
        if (v < n) {
            const int vb = a.vbits[b * n + v];
            bits = ((vb >> 2) ^ vb) & 3;
            d[v] = (uint8_t)bits;
            if (a.x_diff.ptr) a.x_diff(b, v) = bits & 1;
            if (a.z_diff.ptr) a.z_diff(b, v) = (bits >> 1) & 1;
        }
        const uint32_t bx = __ballot_sync(0xffffffffu, bits & 1), bz = __ballot_sync(0xffffffffu, bits & 2);
        if ((tid & 31) == 0) { xw[v >> 5] = bx; zw[v >> 5] = bz; }
    }
    __syncthreads();
    if (a.xd_words) for (int wi = tid; wi < W; wi += T) a.xd_words[b * a.wq + wi] = xw[wi];
    if (a.zd_words) for (int wi = tid; wi < W; wi += T) a.zd_words[b * a.wq + wi] = zw[wi];
    int flagged = 0;
    for (int c = tid; c < a.X.m + a.Z.m; c += T) {
        const bool isx = c < a.X.m;                      // hx checks z_diff (quaternary) / the noise (binary)
        const SideDev &S = isx ? a.X : a.Z;
        const int cc = isx ? c : c - a.X.m;
        const int bit = (isx && !a.binary) ? 1 : 0;
        int par = 0;
        for (int k = S.cn_ptr[cc]; k < S.cn_ptr[cc + 1]; k++) par ^= (d[S.cn_vn[k]] >> bit) & 1;
        flagged |= par;
    }
    // logical operators: any(lz . x_diff) or any(lx . z_diff); one warp per row
    int logical = 0;
    const int warp = tid >> 5, lane = tid & 31, nwarps = T >> 5;
    for (int r = warp; r < a.kx + a.kz; r += nwarps) {
        const bool isz = r >= a.kx;                      // rows of lz act on x_diff
        const uint32_t *row = isz ? a.lz_bits + (int64_t)(r - a.kx) * W : a.lx_bits + (int64_t)r * W;
        const uint32_t *dw = (isz || a.binary) ? xw : zw;
        uint32_t acc = 0;
        for (int wi = lane; wi < W; wi += 32) acc ^= row[wi] & dw[wi];
        acc = __reduce_xor_sync(0xffffffffu, acc);
        logical |= __popc(acc) & 1;
    }
    flagged = __syncthreads_or(flagged);
    logical = __syncthreads_or(logical);
    if (tid == 0) {
        // quaternary: any(hx_perp . d) == flagged or logical.  binary (BP_BSC_Model): ls_hat = logical_pcm . d only
        const int blk = a.binary ? (a.kx > 0 ? logical : flagged) : (flagged | logical);
        const int rnd = a.rounds ? a.rounds[b] : 0;
        if (a.flags) a.flags[b] = (uint8_t)((flagged ? 1 : 0) | (blk ? 2 : 0) | (rnd << 2));
        if (a.frame_bits) {
            const uint32_t bit = 1u << (b & 31);
            if (flagged) atomicOr(a.frame_bits + (b >> 5), bit);
            if (blk) atomicOr(a.frame_bits + a.fw + (b >> 5), bit);
            if (rnd > 0) atomicOr(a.frame_bits + 2 * a.fw + (b >> 5), bit);
        }
        if (a.counters) {
            atomicAdd(a.counters + 0, 1ull);
            if (flagged) atomicAdd(a.counters + 1, 1ull);
            if (blk) atomicAdd(a.counters + 2, 1ull);
            if (rnd > 0) atomicAdd(a.counters + 3, 1ull);
        }
    }
}

// ------------------------------------------------------------------ probes ------------
// Functions of several arguments take them from the input at the element's index and at three others (the same for the
// scalar and the paired form).  Paired forms (fn >= 25) evaluate elements 2i and 2i+1 as the two lanes of one call.
struct ProbeArgs {
    float a0, a1, a2, a3;
    __device__ ProbeArgs(const float *x, int64_t n, int64_t i)
        : a0(x[i]), a1(x[n - 1 - i]), a2(x[(i + n / 3) % n]), a3(x[(i + 2 * (n / 3)) % n]) {}
};
static __global__ void k_math_probe(int fn, const float *x, float *y, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (fn >= 25) {
        if (i & 1) return;
        const int64_t i1 = i + 1 < n ? i + 1 : i;
        const ProbeArgs p(x, n, i), q(x, n, i1);
        const float2 a0 = make_float2(p.a0, q.a0), a1 = make_float2(p.a1, q.a1);
        float2 r;
        switch (fn) {
            case 25: r = fb_sfu_exp2s2(a0, -FB_LOG2E); break;
            case 26: r = fb_sfu_logaddexp_open2(a0, a1); break;
            case 27: r = fb_sfu_vn_corr2(a0, a1); break;
            case 28: r = fb_sfu_vn_msg2(a0, a1, make_float2(p.a2, q.a2), make_float2(p.a3, q.a3)); break;
            case 29: r = fb_sfu_phi_open2(a0); break;
            case 30: r = fb_sfu_softplusf2(a0); break;
            default: r = fb_sfu_tanhf2(a0); break;
        }
        y[i] = r.x;
        if (i1 != i) y[i1] = r.y;
        return;
    }
    const float v = x[i];
    float r;
    const ProbeArgs p(x, n, i);
    switch (fn) {
        case 20: r = fb_sfu_exp2s(v, -FB_LOG2E); break;
        case 21: r = fb_sfu_logaddexp_open(p.a0, p.a1); break;
        case 22: r = fb_sfu_vn_corr(p.a0, p.a1); break;
        case 23: r = fb_sfu_vn_msg(p.a0, p.a1, p.a2, p.a3); break;
        case 24: r = fb_sfu_phi_open(v); break;
        case 0: r = fb_expf(v); break;
        case 1: r = fb_logf(v); break;
        case 2: r = fb_log1pf_pos(v); break;
        case 3: r = fb_softplusf(v); break;
        case 4: r = fb_phi4f(v); break;
        case 5: r = fb_phi2f(v); break;
        case 6: r = fb_tanhf(v); break;
        case 7: r = fb_atanhf(v); break;
        case 8: r = fb_mufu_ex2(v); break;              // raw MUFU.EX2 (tools/dump_sfu_tables.py)
        case 9: r = fb_mufu_lg2(v); break;              // raw MUFU.LG2
        case 15: r = fb_mufu_rcp(v); break;             // raw MUFU.RCP
        case 16: r = fb_sfu_tanhf(v); break;
        case 17: r = fb_sfu_atanhf(v); break;
        case 10: r = fb_sfu_expf(v); break;
        case 11: r = fb_sfu_logf(v); break;
        case 12: r = fb_sfu_softplusf(v); break;
        case 13: r = fb_sfu_phi4f(v); break;
        default: r = fb_sfu_phi2f(v); break;
    }
    y[i] = r;
}

// MUFU throughput: chains of ex2.approx, 8 independent chains per thread
static __global__ void k_sfu_peak(float *out, int iters) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; j++) v[j] = -1.0f - 0.001f * (float)(threadIdx.x + j);
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 8; j++) asm volatile("ex2.approx.ftz.f32 %0, %0;" : "+f"(v[j]));
    }
    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; j++) s += v[j];
    if (s == 123.456f) out[0] = s;
}

// FP32 FMA issue rate: 8 independent FFMA chains per thread
static __global__ void k_fma_peak(float *out, int iters) {
    float v[8];
    const float a = 0.999f + 1e-6f * (float)threadIdx.x, c = 1e-3f;
#pragma unroll
    for (int j = 0; j < 8; j++) v[j] = 0.5f + 0.01f * (float)j;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 8; j++) v[j] = __fmaf_rn(v[j], a, c);
    }
    float s = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; j++) s += v[j];
    if (s == 123.456f) out[0] = s;
}

static __global__ void k_fill(uint32_t *p, int64_t n, uint32_t v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        p[i] = v;
}

}  // namespace fbgnn
