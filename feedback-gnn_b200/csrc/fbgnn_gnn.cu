// fbgnn_gnn.cu -- feedback GNN: weight packing, launch selection, C ABI.
#include "fbgnn_internal.h"
#include "fbgnn_gnn_tc.cuh"

// ------------------------------------------------------------------ feedback GNN --------
template <int H, int M>
static void pack_gnn(std::vector<float> &w, const float *W0, const float *b0, const float *W1x,
                     const float *b1x, const float *W2x, const float *b2x, const float *W1z,
                     const float *b1z, const float *W2z, const float *b2z, const float *W3, const float *b3) {
    typedef GnnLayout<H, M> L;
    w.assign(L::total, 0.0f);
    auto put = [&](int off, const float *src, int count) { if (src) std::memcpy(&w[off], src, sizeof(float) * count); };
    put(L::W1x, W1x, 4 * H); put(L::b1x, b1x, H); put(L::W2x, W2x, H * M); put(L::b2x, b2x, M);
    put(L::W1z, W1z, 4 * H); put(L::b1z, b1z, H); put(L::W2z, W2z, H * M); put(L::b2z, b2z, M);
    put(L::W3, W3, (2 * M + 3) * H); put(L::b3, b3, H); put(L::W0, W0, H * 3); put(L::b0, b0, 3);
    for (int j = 0; j < H; j++)
        for (int k = 0; k < 4; k++) {
            w[L::W1tx + 4 * j + k] = W1x[k * H + j];
            w[L::W1tz + 4 * j + k] = W1z[k * H + j];
        }
}

extern "C" int fbgnn_gnn_create(fbgnn_ctx *ctx, int32_t H, int32_t M, int32_t activation, int32_t reduce_op,
                                const float *W0, const float *b0, const float *W1x, const float *b1x,
                                const float *W2x, const float *b2x, const float *W1z, const float *b1z,
                                const float *W2z, const float *b2z, const float *W3, const float *b3,
                                fbgnn_gnn **out) {
    REQUIRE(ctx && out, "NULL argument");
    REQUIRE(W0 && W1x && W2x && W1z && W2z && W3, "weight matrices must not be NULL");
    REQUIRE(activation >= 0 && activation <= 2, "unknown activation %d", activation);
    REQUIRE(reduce_op >= 0 && reduce_op <= 3, "unknown reduce_op %d", reduce_op);
    const bool any_b = b0 || b1x || b2x || b1z || b2z || b3, all_b = b0 && b1x && b2x && b1z && b2z && b3;
    REQUIRE(any_b == all_b, "either all biases or none must be given");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    std::vector<float> w;
    if (H == 40 && M == 20) pack_gnn<40, 20>(w, W0, b0, W1x, b1x, W2x, b2x, W1z, b1z, W2z, b2z, W3, b3);
    else if (H == 20 && M == 20) pack_gnn<20, 20>(w, W0, b0, W1x, b1x, W2x, b2x, W1z, b1z, W2z, b2z, W3, b3);
    else if (H == 64 && M == 32) pack_gnn<64, 32>(w, W0, b0, W1x, b1x, W2x, b2x, W1z, b1z, W2z, b2z, W3, b3);
    else return fail(FBGNN_E_UNSUPPORTED, "Feedback_GNN with num_hidden_units=%d, num_msg_dims=%d is not "
                     "compiled into this build (available: 40/20, 20/20, 64/32)", H, M);
    fbgnn_gnn *g = new fbgnn_gnn();
    g->ctx = ctx; g->H = H; g->M = M; g->act = activation; g->reduce = reduce_op; g->use_bias = all_b ? 1 : 0;
    g->total = (int)w.size();
    CK(cudaMalloc(&g->weights, w.size() * sizeof(float)));
    CK(cudaMemcpy(g->weights, w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice));
    if (H == 40 && M == 20) {   // tensor-core operand tiles (TF32 hi / lo, canonical K-major UMMA layout) + the scalar block
        using tc::GnnW;
        std::vector<float> tv(GnnW::total, 0.0f);
        auto tile = [&](int off, int kpad, int npad, auto wf) {
            for (int nn = 0; nn < npad; nn++)
                for (int k = 0; k < kpad; k++) {
                    const float x = wf(k, nn), hi = tc::tf32_hi(x);
                    tv[off + tc::b_tile_offset(nn, k, kpad)] = hi;
                    tv[off + kpad * npad + tc::b_tile_offset(nn, k, kpad)] = x - hi;
                }
        };
        // reduce_op mean: the division by the node degree (3: this form is built for (3,.)-regular codes) is folded into
        // the tiles as a multiplication by float32(1/3); the oracle's tensor-core form scales W2 the same way
        const float inv = reduce_op == 0 ? 1.0f / 3.0f : 1.0f;
        tile(GnnW::W2X, 40, 32, [&](int k, int nn) { return nn < 20 ? W2x[k * 20 + nn] * inv : 0.0f; });
        tile(GnnW::W2Z, 40, 32, [&](int k, int nn) { return nn < 20 ? W2z[k * 20 + nn] * inv : 0.0f; });
        tile(GnnW::W3AB, 40, 48, [&](int k, int nn) { return nn < 40 ? W3[k * 40 + nn] : 0.0f; });
        std::memcpy(&tv[GnnW::SCALAR], w.data(), sizeof(float) * w.size());
        // first-layer rows of hidden units j, j+1 interleaved (k_gnn_tc's edge phase evaluates them as a pair)
        typedef GnnLayout<40, 20> L;
        for (int j = 0; j < 40; j++)
            for (int k = 0; k < 4; k++) {
                tv[GnnW::SCALAR + L::W1tx + 8 * (j >> 1) + 2 * k + (j & 1)] = W1x[k * 40 + j];
                tv[GnnW::SCALAR + L::W1tz + 8 * (j >> 1) + 2 * k + (j & 1)] = W1z[k * 40 + j];
            }
        CK(cudaMalloc(&g->w_tc, tv.size() * sizeof(float)));
        CK(cudaMemcpy(g->w_tc, tv.data(), tv.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    *out = g;
    return 0;
}

extern "C" int fbgnn_gnn_set_gemm(fbgnn_gnn *g, int32_t mode) {
    REQUIRE(g, "NULL handle");
    REQUIRE(mode == FBGNN_GEMM_FMA || mode == FBGNN_GEMM_TF32X3, "unknown gemm mode %d", mode);
    if (mode == FBGNN_GEMM_TF32X3 && !(g->w_tc && g->layers == 2 && g->reduce <= 1 && g->act == FBGNN_ACT_TANH))
        return fail(FBGNN_E_UNSUPPORTED, "the tensor-core form of the feedback GNN is built for num_hidden_units = 40, "
                    "num_msg_dims = 20, 2-layer MLPs, tanh, reduce_op mean / sum");
    g->gemm = mode;
    return 0;
}

extern "C" int fbgnn_umma_probe(fbgnn_ctx *ctx, const float *A, const float *B, const float *Din, float *Dout, int32_t trials) {
    REQUIRE(ctx && A && B && Din && Dout && trials >= 0, "bad argument");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    if (trials == 0) return 0;
    tc::k_umma_probe<<<1, 128, 0, ctx->stream>>>(A, B, Din, Dout, trials);
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}

extern "C" int fbgnn_gnn_create_deep(fbgnn_ctx *ctx, int32_t H, int32_t M, int32_t num_mlp_layers, int32_t activation,
                                     int32_t reduce_op, int32_t use_bias, const float *packed, int64_t count,
                                     fbgnn_gnn **out) {
    REQUIRE(ctx && out && packed, "NULL argument");
    REQUIRE(H >= 1 && H <= GNND_MAX && M >= 1 && M <= GNND_MAX, "hidden / message dims must be in [1, %d]", GNND_MAX);
    REQUIRE(num_mlp_layers >= 1 && num_mlp_layers <= 8, "num_mlp_layers must be in [1, 8]");
    REQUIRE(activation >= 0 && activation <= 2 && reduce_op >= 0 && reduce_op <= 3, "bad activation / reduce_op");
    const int L = num_mlp_layers;
    int64_t want = (int64_t)(L == 1 ? 2 * M + 3 : H) * 3 + 3;
    {
        int kin = 4;
        int64_t side = 0;
        for (int l = 0; l < L; l++) { const int kout = (l == L - 1) ? M : H; side += (int64_t)kin * kout + kout; kin = kout; }
        want += 2 * side;
        kin = 2 * M + 3;
        for (int l = 0; l < L - 1; l++) { want += (int64_t)kin * H + H; kin = H; }
    }
    REQUIRE(count == want, "packed weights hold %lld floats, the layer sequence needs %lld", (long long)count, (long long)want);
    if (set_device(ctx)) return FBGNN_E_CUDA;
    fbgnn_gnn *g = new fbgnn_gnn();
    g->ctx = ctx; g->H = H; g->M = M; g->act = activation; g->reduce = reduce_op; g->use_bias = use_bias ? 1 : 0;
    g->layers = L; g->total = (int)count;
    CK(cudaMalloc(&g->weights, (size_t)count * sizeof(float)));
    CK(cudaMemcpy(g->weights, packed, (size_t)count * sizeof(float), cudaMemcpyHostToDevice));
    *out = g;
    return 0;
}

extern "C" int fbgnn_gnn_destroy(fbgnn_gnn *g) {
    if (!g) return 0;
    cudaSetDevice(g->ctx->device);
    cudaStreamSynchronize(g->ctx->stream);
    cudaFree(g->weights);
    cudaFree(g->w_tc);
    delete g;
    return 0;
}

template <int H, int M, int DV, bool TB, bool FACT, typename MATH>
static int launch_gnn_t(fbgnn_ctx *ctx, const GnnArgs &a) {
    const size_t smem = sizeof(float) * GnnLayout<H, M>::total;
    if (int rc = set_smem(k_gnn<H, M, DV, TB, FACT, MATH>, smem, ctx, "feedback GNN")) return rc;
    const int64_t items = a.num_frames * a.X.n;
    int64_t blocks = (items + 127) / 128;
    blocks = std::min<int64_t>(blocks, (int64_t)ctx->num_sms * 8);
    k_gnn<H, M, DV, TB, FACT, MATH><<<(unsigned)blocks, 128, smem, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}

template <int H, int M, int DV, bool TB, bool FACT = true>
static int launch_gnn_m(fbgnn_ctx *ctx, const GnnArgs &a) {
    return ctx->math_mode == FBGNN_MATH_SFU ? launch_gnn_t<H, M, DV, TB, FACT, MathSfu>(ctx, a)
                                             : launch_gnn_t<H, M, DV, TB, FACT, MathExact>(ctx, a);
}

int launch_gnn(fbgnn_ctx *ctx, const fbgnn_gnn *g, GnnArgs &a) {
    if (a.num_frames <= 0) return 0;
    a.weights = g->weights; a.act = g->act; a.reduce = g->reduce; a.use_bias = g->use_bias;
    if (g->layers != 2) {                      // general depth: k_gnn_deep
        GnnDeepArgs d{a, g->H, g->M, g->layers};
        const int64_t items = a.num_frames * a.X.n;
        const unsigned blocks = (unsigned)std::min<int64_t>((items + 127) / 128, (int64_t)ctx->num_sms * 16);
        if (ctx->math_mode == FBGNN_MATH_SFU) k_gnn_deep<MathSfu><<<blocks, 128, 0, ctx->stream>>>(d);
        else k_gnn_deep<MathExact><<<blocks, 128, 0, ctx->stream>>>(d);
        CK(cudaGetLastError());
        ctx->launches++;
        return 0;
    }
    const bool reg3 = a.X.reg_dv == 3 && a.Z.reg_dv == 3;      // the (3,6)-regular GHP / bivariate codes
    if (g->gemm == FBGNN_GEMM_TF32X3) {                         // opt-in: dense products on tcgen05 (fbgnn_gnn_tc.cuh)
        if (!reg3) return fail(FBGNN_E_UNSUPPORTED, "the tensor-core form of the feedback GNN needs (3, .)-regular sides");
        const size_t smem = sizeof(float) * tc::GnnW::total;
        const int64_t tiles = (a.num_frames * a.X.n + 127) / 128;
        const unsigned blocks = (unsigned)std::min<int64_t>((tiles + 1) / 2, (int64_t)ctx->num_sms * 2);
        if (ctx->math_mode == FBGNN_MATH_SFU) {
            if (int rc = set_smem(tc::k_gnn_tc<3, MathSfu>, smem, ctx, "feedback GNN (tensor cores)")) return rc;
            tc::k_gnn_tc<3, MathSfu><<<blocks, 256, smem, ctx->stream>>>(a, g->w_tc);
        } else {
            if (int rc = set_smem(tc::k_gnn_tc<3, MathExact>, smem, ctx, "feedback GNN (tensor cores)")) return rc;
            tc::k_gnn_tc<3, MathExact><<<blocks, 256, smem, ctx->stream>>>(a, g->w_tc);
        }
        CK(cudaGetLastError());
        ctx->launches++;
        return 0;
    }
    const bool tb = g->act == FBGNN_ACT_TANH && g->use_bias;   // the shipped configuration
    const bool fact = g->reduce <= 1;                          // mean / sum: output layer after the reduction
    if (g->H == 40 && g->M == 20) {
        if (!fact) return launch_gnn_m<40, 20, 0, false, false>(ctx, a);
        if (reg3 && tb) return launch_gnn_m<40, 20, 3, true>(ctx, a);
        if (reg3) return launch_gnn_m<40, 20, 3, false>(ctx, a);
        return tb ? launch_gnn_m<40, 20, 0, true>(ctx, a) : launch_gnn_m<40, 20, 0, false>(ctx, a);
    }
    if (g->H == 20 && g->M == 20) return fact ? launch_gnn_m<20, 20, 0, false>(ctx, a) : launch_gnn_m<20, 20, 0, false, false>(ctx, a);
    if (g->H == 64 && g->M == 32) return fact ? launch_gnn_m<64, 32, 0, false>(ctx, a) : launch_gnn_m<64, 32, 0, false, false>(ctx, a);
    return fail(FBGNN_E_UNSUPPORTED, "unsupported GNN dimensions");
}

extern "C" int fbgnn_gnn_forward(fbgnn_code *code, fbgnn_gnn *gnn, int64_t B, fbgnn_tensor3 h_vn,
                                 fbgnn_tensor2 logit_hx, fbgnn_tensor2 logit_hz, fbgnn_tensor2 synd_x,
                                 fbgnn_tensor2 synd_z, fbgnn_tensor3 out) {
    REQUIRE(code && gnn, "NULL handle");
    REQUIRE(h_vn.ptr && logit_hx.ptr && logit_hz.ptr && synd_x.ptr && synd_z.ptr && out.ptr, "NULL tensor");
    REQUIRE(B >= 0, "B must be non-negative");
    fbgnn_ctx *ctx = code->ctx;
    if (set_device(ctx)) return FBGNN_E_CUDA;
    GnnArgs a{};
    a.X = code->X->dev; a.Z = code->Z->dev;
    a.num_frames = B;
    a.h_vn = v3<const float>(h_vn);
    a.logit_hx = v2<const float>(logit_hx); a.logit_hz = v2<const float>(logit_hz);
    a.sx = v2<const uint8_t>(synd_x); a.sz = v2<const uint8_t>(synd_z);
    a.out = v3<float>(out);
    return launch_gnn(ctx, gnn, a);
}

