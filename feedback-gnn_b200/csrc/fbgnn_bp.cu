// fbgnn_bp.cu -- launch configuration of the BP kernels and the decoder entry points of the C ABI.
#include "fbgnn_internal.h"
#include "fbgnn_cluster.cuh"

// ------------------------------------------------------------------ launch helpers ------
// Threads per CTA for the one-frame-per-CTA kernels: the multiple of 32 in [128, 512] that
// wastes the fewest lanes over the variable-node and check-node passes.
static int pick_threads(int n_items_a, int n_items_b) {
    auto eff = [&](int t) {
        const double pa = (double)((n_items_a + t - 1) / t) * t, pb = (double)((n_items_b + t - 1) / t) * t;
        return (double)(n_items_a + n_items_b) / (pa + pb);
    };
    int best = 256;
    for (int t = 128; t <= 512; t += 32)
        if (eff(t) > eff(best) + 0.004) best = t;      // keep 256 unless another size is clearly better
    return best;
}

static size_t bp4_smem(const SideDev &X, const SideDev &Z, bool const_prior, bool iter_logits) {
    const size_t np = (size_t)pad4(X.n);
    return sizeof(float) * ((size_t)X.E + Z.E + ((const_prior ? 2 : 3) + (iter_logits ? 2 : 0)) * np) +
           (size_t)pad16(X.m + Z.m) + 2 * (((size_t)X.n + 1) & ~(size_t)1) + X.n + 16;
}

template <bool CP, int DV, int DC, typename MATH, bool FPX>
static int launch_bp4_t(fbgnn_ctx *ctx, const Bp4Args &a, int64_t grid, size_t smem, int threads) {
    if (int rc = set_smem(k_bp4<CP, DV, DC, MATH, FPX>, smem, ctx, "quaternary BP")) return rc;
    k_bp4<CP, DV, DC, MATH, FPX><<<(unsigned)grid, threads, smem, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}

template <int DV, int DC>
static int launch_bp4_m(fbgnn_ctx *ctx, const Bp4Args &a, int64_t grid, size_t smem, int threads, bool cp) {
    // fixed-point exit: regular graph, boxplus-phi, long runs (the bookkeeping costs ~5 % per unsaturated iteration
    // and a 16-iteration stage does not converge-and-saturate in time).  Valid in both arithmetics: the saturation
    // constants are exact in each.  From 32 iterations on: with the exit in the 16-iteration stages too, the headline
    // pipeline measured 430.7 k instead of 441.1 k frames/s on B200 (profiles/r02_lab_k_bp4_variants.txt).
    const bool fpx = DV > 0 && a.cn_type == 0 && a.num_iter >= 32 && !a.iter_logits.ptr;
    if (ctx->math_mode == FBGNN_MATH_SFU) {
        if (fpx)
            return cp ? launch_bp4_t<true, DV, DC, MathSfu, true>(ctx, a, grid, smem, threads)
                      : launch_bp4_t<false, DV, DC, MathSfu, true>(ctx, a, grid, smem, threads);
        return cp ? launch_bp4_t<true, DV, DC, MathSfu, false>(ctx, a, grid, smem, threads)
                  : launch_bp4_t<false, DV, DC, MathSfu, false>(ctx, a, grid, smem, threads);
    }
    if (fpx)
        return cp ? launch_bp4_t<true, DV, DC, MathExact, true>(ctx, a, grid, smem, threads)
                  : launch_bp4_t<false, DV, DC, MathExact, true>(ctx, a, grid, smem, threads);
    return cp ? launch_bp4_t<true, DV, DC, MathExact, false>(ctx, a, grid, smem, threads)
              : launch_bp4_t<false, DV, DC, MathExact, false>(ctx, a, grid, smem, threads);
}

// Codes whose per-frame state does not fit the shared memory of an SM: generic kernel with the float arrays in HBM.
template <typename MATH>
static int launch_bp4_gstate(fbgnn_ctx *ctx, Bp4Args a, int64_t grid, int threads, bool cp) {
    const SideDev &X = a.X, &Z = a.Z;
    const size_t smem = (size_t)pad16(X.m + Z.m) + 2 * (((size_t)X.n + 1) & ~(size_t)1) + X.n + 16;
    a.state_stride = (int64_t)X.E + Z.E + ((cp ? 2 : 3) + (a.iter_logits.ptr ? 2 : 0)) * (int64_t)pad4(X.n);
    CK(cudaMallocAsync(&a.state, sizeof(float) * (size_t)grid * a.state_stride, ctx->stream));
    int rc;
    if (cp) {
        rc = set_smem(k_bp4<true, 0, 0, MATH, false, true>, smem, ctx, "quaternary BP (HBM state)");
        if (!rc) k_bp4<true, 0, 0, MATH, false, true><<<(unsigned)grid, threads, smem, ctx->stream>>>(a);
    } else {
        rc = set_smem(k_bp4<false, 0, 0, MATH, false, true>, smem, ctx, "quaternary BP (HBM state)");
        if (!rc) k_bp4<false, 0, 0, MATH, false, true><<<(unsigned)grid, threads, smem, ctx->stream>>>(a);
    }
    CK(cudaFreeAsync(a.state, ctx->stream));
    if (rc) return rc;
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}

// Codes beyond one SM's shared memory, fast path: a thread-block cluster of 2 / 4 / 8 CTAs per frame with the messages in
// distributed shared memory (fbgnn_cluster.cuh).  Returns 1 if the configuration is not served (caller falls back).
template <bool CP, typename MATH, int DCMAX>
static int launch_bp4_cluster_t(fbgnn_ctx *ctx, const Bp4Args &a, int64_t frames, const ClusterPart &P, size_t smem) {
    auto kernel = k_bp4_cluster<CP, MATH, DCMAX>;
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(frames * P.C), 1, 1);
    cfg.blockDim = dim3(512, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)P.C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    CK(cudaLaunchKernelEx(&cfg, kernel, a, P));
    ctx->launches++;
    return 0;
}

template <bool CP, typename MATH>
static int launch_bp4_cluster_d(fbgnn_ctx *ctx, const Bp4Args &a, int64_t frames, const ClusterPart &P, size_t smem, int max_dc) {
    return max_dc <= 8 ? launch_bp4_cluster_t<CP, MATH, 8>(ctx, a, frames, P, smem)
                       : launch_bp4_cluster_t<CP, MATH, 64>(ctx, a, frames, P, smem);
}

static int launch_bp4_cluster(fbgnn_ctx *ctx, const Bp4Args &a, int64_t frames, bool cp, int max_dc) {
    const SideDev &X = a.X, &Z = a.Z;
    if (!X.h_vn_ptr || !Z.h_vn_ptr || a.iter_logits.ptr || a.iters_out || a.rows_x_ptr) return 1;
    const int n = X.n, mt = X.m + Z.m;
    // Smallest cluster of at least 4 CTAs whose CTAs fit: 4 CTAs per frame measured best on the [[7688,50]] code (2: too
    // few warps per SM; 8: barrier cost; profiles/r02_cluster_vs_gstate.txt).
    for (int C = 4; C <= CL_MAX; C *= 2) {
        ClusterPart P{};
        P.C = C;
        for (int r = 0; r <= C; r++) {
            P.v0[r] = (int)((int64_t)n * r / C);
            P.ex0[r] = X.h_vn_ptr[P.v0[r]];
            P.ez0[r] = Z.h_vn_ptr[P.v0[r]];
            P.c0[r] = (int)((int64_t)mt * r / C);
        }
        for (int r = 0; r < C; r++) {
            P.nv_max = std::max(P.nv_max, P.v0[r + 1] - P.v0[r]);
            P.ex_max = std::max(P.ex_max, P.ex0[r + 1] - P.ex0[r]);
            P.ez_max = std::max(P.ez_max, P.ez0[r + 1] - P.ez0[r]);
        }
        const size_t smem = sizeof(float) * ((size_t)P.ex_max + P.ez_max + (cp ? 2 : 3) * (size_t)P.nv_max) +
                            (((size_t)P.nv_max + 3) & ~(size_t)3) + sizeof(int) * CL_MAX;
        if (smem > ctx->smem_optin) continue;
        if (ctx->math_mode == FBGNN_MATH_SFU)
            return cp ? launch_bp4_cluster_d<true, MathSfu>(ctx, a, frames, P, smem, max_dc) : launch_bp4_cluster_d<false, MathSfu>(ctx, a, frames, P, smem, max_dc);
        return cp ? launch_bp4_cluster_d<true, MathExact>(ctx, a, frames, P, smem, max_dc) : launch_bp4_cluster_d<false, MathExact>(ctx, a, frames, P, smem, max_dc);
    }
    return 1;
}

int launch_bp4(fbgnn_ctx *ctx, const Bp4Args &a_in, int64_t grid) {
    if (grid <= 0) return 0;
    Bp4Args a = a_in;
    a.stats = ctx->stats;
    const bool cp = a.llr.ptr == nullptr;
    const size_t smem = bp4_smem(a.X, a.Z, cp, a.iter_logits.ptr != nullptr);
    const int threads = pick_threads(a.X.n, a.X.m + a.Z.m);
    if (smem > ctx->smem_optin) {
        // Larger than one SM: a thread-block cluster with the messages in distributed shared memory, or the kernel whose
        // state lives in HBM / L2.  Measured on the [[7688,50]] code (profiles/r02_cluster_vs_gstate.txt): the cluster of
        // 4 wins by 7 % in exact arithmetic, the L2-state kernel by 17 % in SFU arithmetic (its state stays L2-resident
        // and it keeps more warps per SM) -- the default follows the measurement, FBGNN_BP4_LARGE=cluster|gstate overrides.
        const char *force = getenv("FBGNN_BP4_LARGE");
        const bool want_cluster = force ? !strcmp(force, "cluster") : ctx->math_mode != FBGNN_MATH_SFU;
        if (want_cluster) {
            const int max_dc = (a.X.reg_dc && a.Z.reg_dc) ? std::max(a.X.reg_dc, a.Z.reg_dc) : 64;
            const int rc = launch_bp4_cluster(ctx, a, grid, cp, max_dc);
            if (rc <= 0) return rc;
        }
        return ctx->math_mode == FBGNN_MATH_SFU ? launch_bp4_gstate<MathSfu>(ctx, a, grid, threads, cp)
                                                 : launch_bp4_gstate<MathExact>(ctx, a, grid, threads, cp);
    }
    // both sides regular with the same degrees -> unrolled instantiation
    int dv = 0, dc = 0;
    if (a.X.reg_dv && a.X.reg_dv == a.Z.reg_dv && a.X.reg_dc && a.X.reg_dc == a.Z.reg_dc) { dv = a.X.reg_dv; dc = a.X.reg_dc; }
    if (dv == 3 && dc == 6) return launch_bp4_m<3, 6>(ctx, a, grid, smem, threads, cp);
    if (dv == 4 && dc == 8) return launch_bp4_m<4, 8>(ctx, a, grid, smem, threads, cp);
    if (dv == 5 && dc == 10) return launch_bp4_m<5, 10>(ctx, a, grid, smem, threads, cp);
    return launch_bp4_m<0, 0>(ctx, a, grid, smem, threads, cp);
}

// ------------------------------------------------------------------ decoders ------------
extern "C" int fbgnn_rows_create(fbgnn_ctx *ctx, int32_t n, int32_t m, const int32_t *indptr, const int32_t *indices,
                                 fbgnn_rows **out) {
    REQUIRE(ctx && out && indptr, "NULL argument");
    REQUIRE(n > 0 && n <= 65535 && m >= 0, "bad shape (%d x %d; at most 65535 columns)", m, n);
    REQUIRE(indptr[0] == 0, "indptr[0] != 0");
    for (int r = 0; r < m; r++) {
        REQUIRE(indptr[r + 1] >= indptr[r], "indptr not monotone at row %d", r);
        for (int k = indptr[r]; k < indptr[r + 1]; k++)
            REQUIRE(indices[k] >= 0 && indices[k] < n, "column index out of range in row %d", r);
    }
    if (set_device(ctx)) return FBGNN_E_CUDA;
    fbgnn_rows *R = new fbgnn_rows();
    R->ctx = ctx; R->n = n; R->m = m;
    std::vector<idx_t> col(std::max(indptr[m], 1));
    for (int k = 0; k < indptr[m]; k++) col[k] = (idx_t)indices[k];
    CK(cudaMalloc(&R->ptr, sizeof(int) * (size_t)(m + 1)));
    CK(cudaMemcpy(R->ptr, indptr, sizeof(int) * (size_t)(m + 1), cudaMemcpyHostToDevice));
    CK(cudaMalloc(&R->col, sizeof(idx_t) * col.size()));
    CK(cudaMemcpy(R->col, col.data(), sizeof(idx_t) * col.size(), cudaMemcpyHostToDevice));
    *out = R;
    return 0;
}

extern "C" int fbgnn_rows_destroy(fbgnn_rows *R) {
    if (!R) return 0;
    cudaSetDevice(R->ctx->device);
    cudaFree(R->ptr); cudaFree(R->col);
    delete R;
    return 0;
}

extern "C" int fbgnn_bp4_decode_ex(fbgnn_code *code, int32_t cn_type, int32_t num_iter, float factor, int64_t B,
                                   fbgnn_tensor3 llr, float prior, fbgnn_tensor2 synd_x, fbgnn_tensor2 synd_z,
                                   fbgnn_tensor2 Lx, fbgnn_tensor2 Ly, fbgnn_tensor2 Lz, fbgnn_tensor2 x_hat,
                                   fbgnn_tensor2 z_hat, fbgnn_tensor2 x_logit, fbgnn_tensor2 z_logit,
                                   fbgnn_tensor2 msg_x, fbgnn_tensor2 msg_z, fbgnn_tensor3 iter_logits,
                                   const fbgnn_bp4_opts *opts) {
    REQUIRE(code, "code is NULL");
    REQUIRE(cn_type >= 0 && cn_type <= 2, "unknown cn_type %d", cn_type);
    REQUIRE(num_iter >= 0 && B >= 0, "num_iter and B must be non-negative");
    REQUIRE(synd_x.ptr && synd_z.ptr, "syndromes are NULL");
    fbgnn_ctx *ctx = code->ctx;
    if (set_device(ctx)) return FBGNN_E_CUDA;
    Bp4Args a{};
    a.X = code->X->dev; a.Z = code->Z->dev;
    a.cn_type = cn_type; a.num_iter = num_iter; a.factor = factor;
    a.llr = v3<const float>(llr); a.prior = prior;
    a.sx = v2<const uint8_t>(synd_x); a.sz = v2<const uint8_t>(synd_z);
    a.Lx = v2<float>(Lx); a.Ly = v2<float>(Ly); a.Lz = v2<float>(Lz);
    a.xh = v2<uint8_t>(x_hat); a.zh = v2<uint8_t>(z_hat);
    a.xl = v2<float>(x_logit); a.zl = v2<float>(z_logit);
    a.msg_x = v2<float>(msg_x); a.msg_z = v2<float>(msg_z);
    a.iter_logits = v3<float>(iter_logits);
    if (opts) {
        REQUIRE(!opts->iters_out || num_iter <= 255, "early stop reports iteration counts as uint8 (num_iter <= 255)");
        REQUIRE(!opts->iters_out || !iter_logits.ptr, "early stop and per-iteration soft syndromes exclude each other");
        REQUIRE((opts->rows_x == nullptr) == (opts->rows_z == nullptr), "give both rows_x and rows_z or neither");
        a.iters_out = opts->iters_out;
        if (opts->rows_x) {
            REQUIRE(opts->rows_x->n == a.X.n && opts->rows_z->n == a.X.n, "row sets must have n = %d columns", a.X.n);
            a.rows_x_ptr = opts->rows_x->ptr; a.rows_x_col = opts->rows_x->col; a.rows_x_m = opts->rows_x->m;
            a.rows_z_ptr = opts->rows_z->ptr; a.rows_z_col = opts->rows_z->col; a.rows_z_m = opts->rows_z->m;
        }
    }
    return launch_bp4(ctx, a, B);
}

extern "C" int fbgnn_bp4_decode(fbgnn_code *code, int32_t cn_type, int32_t num_iter, float factor, int64_t B,
                                fbgnn_tensor3 llr, float prior, fbgnn_tensor2 synd_x, fbgnn_tensor2 synd_z,
                                fbgnn_tensor2 Lx, fbgnn_tensor2 Ly, fbgnn_tensor2 Lz, fbgnn_tensor2 x_hat,
                                fbgnn_tensor2 z_hat, fbgnn_tensor2 x_logit, fbgnn_tensor2 z_logit,
                                fbgnn_tensor2 msg_x, fbgnn_tensor2 msg_z, fbgnn_tensor3 iter_logits) {
    return fbgnn_bp4_decode_ex(code, cn_type, num_iter, factor, B, llr, prior, synd_x, synd_z, Lx, Ly, Lz, x_hat, z_hat,
                               x_logit, z_logit, msg_x, msg_z, iter_logits, nullptr);
}

static size_t bp2_smem(const SideDev &S) { return sizeof(float) * ((size_t)S.E + S.n) + S.m + S.n + 16; }

template <int DV, int DC, typename MATH>
static int launch_bp2_t(fbgnn_ctx *ctx, const Bp2Args &a, int64_t B, size_t smem) {
    if (int rc = set_smem(k_bp2<DV, DC, MATH>, smem, ctx, "binary BP")) return rc;
    k_bp2<DV, DC, MATH><<<(unsigned)B, pick_threads(a.S.n, a.S.m), smem, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}

template <int DV, int DC>
static int launch_bp2_m(fbgnn_ctx *ctx, const Bp2Args &a, int64_t B, size_t smem) {
    return ctx->math_mode == FBGNN_MATH_SFU ? launch_bp2_t<DV, DC, MathSfu>(ctx, a, B, smem)
                                             : launch_bp2_t<DV, DC, MathExact>(ctx, a, B, smem);
}

int launch_bp2(fbgnn_ctx *ctx, const Bp2Args &a, int64_t B) {
    if (B <= 0) return 0;
    const size_t smem = bp2_smem(a.S);
    if (a.S.reg_dv == 3 && a.S.reg_dc == 6) return launch_bp2_m<3, 6>(ctx, a, B, smem);
    if (a.S.reg_dv == 4 && a.S.reg_dc == 8) return launch_bp2_m<4, 8>(ctx, a, B, smem);
    if (a.S.reg_dv == 5 && a.S.reg_dc == 10) return launch_bp2_m<5, 10>(ctx, a, B, smem);
    return launch_bp2_m<0, 0>(ctx, a, B, smem);
}

extern "C" int fbgnn_bp2_decode_ex(fbgnn_graph *g, int32_t cn_type, int32_t num_iter, float factor, int64_t B,
                                   fbgnn_tensor2 llr, fbgnn_tensor2 synd, fbgnn_tensor2 soft, fbgnn_tensor2 hard,
                                   const float *edge_weights, fbgnn_tensor2 msg_in, fbgnn_tensor2 msg_out) {
    REQUIRE(g, "graph is NULL");
    REQUIRE(cn_type >= 0 && cn_type <= 2, "unknown cn_type %d", cn_type);
    REQUIRE(num_iter >= 0 && B >= 0, "num_iter and B must be non-negative");
    REQUIRE(llr.ptr, "llr is NULL");
    REQUIRE(soft.ptr || hard.ptr, "no output requested");
    if (int rc = need_decodable(g)) return rc;
    fbgnn_ctx *ctx = g->ctx;
    if (set_device(ctx)) return FBGNN_E_CUDA;
    Bp2Args a{};
    a.S = g->dev; a.cn_type = cn_type; a.num_iter = num_iter; a.factor = factor;
    a.llr = v2<const float>(llr); a.synd = v2<const uint8_t>(synd);
    a.soft = v2<float>(soft); a.hard = v2<uint8_t>(hard);
    a.edge_w = edge_weights;
    a.msg_in = v2<const float>(msg_in); a.msg_out = v2<float>(msg_out);
    return launch_bp2(ctx, a, B);
}

extern "C" int fbgnn_bp2_decode(fbgnn_graph *g, int32_t cn_type, int32_t num_iter, float factor, int64_t B,
                                fbgnn_tensor2 llr, fbgnn_tensor2 synd, fbgnn_tensor2 soft, fbgnn_tensor2 hard) {
    const fbgnn_tensor2 none = {nullptr, 0, 0};
    return fbgnn_bp2_decode_ex(g, cn_type, num_iter, factor, B, llr, synd, soft, hard, nullptr, none, none);
}
