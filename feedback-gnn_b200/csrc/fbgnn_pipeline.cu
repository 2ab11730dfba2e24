// fbgnn_pipeline.cu -- the fused Monte-Carlo pipelines (multi-launch orchestration) and OSD.
#include "fbgnn_internal.h"
#include "fbgnn_osd_cluster.cuh"
#include "fbgnn_lsd.cuh"

// ------------------------------------------------------------------ OSD -----------------
// Dynamic shared memory of one OSD CTA that holds `rows` basis rows; with `cluster`, the layout of k_osd_cluster (its
// slots after the u16 arrays, and csum[n] after cv / sv).  Sets a.cv_off (order > 0) and *slot_off.
static size_t osd_smem(OsdArgs &a, int rows, bool cluster, int *slot_off) {
    const int n = a.S.n, R = a.S.m, W = (n + 1 + 31) / 32, Rp = rows | 1;
    const size_t main_bytes = std::max<size_t>((size_t)a.npad * 8, (size_t)W * Rp * 4);
    const size_t u16_bytes = sizeof(uint16_t) * (2 * (size_t)n + R);
    size_t smem = ((main_bytes + 7) & ~(size_t)7) + u16_bytes + 16;
    size_t cs_base = ((main_bytes + 7) & ~(size_t)7) + ((u16_bytes + 15) & ~(size_t)15);
    if (cluster) {              // slot[2][W + 1], row[W + 1], svl[rows / 32]
        *slot_off = (int)cs_base;
        smem = cs_base + sizeof(uint32_t) * (3 * ((size_t)W + 1) + (size_t)rows / 32);
        cs_base = (smem + 15) & ~(size_t)15;
    }
    if (a.order > 0) {          // OSD-CS: the first lp non-pivot columns and s' as ceil(R/32)-word bit vectors
        const size_t lp = (size_t)std::min(a.order, std::max(n - R, 0)), RW = ((size_t)R + 31) / 32;
        a.cv_off = (int)cs_base;
        smem = cs_base + (lp + 1) * RW * 4 + (cluster ? sizeof(int) * (size_t)n : 0);
    }
    return smem;
}

int launch_osd(fbgnn_ctx *ctx, OsdArgs &a, int order, int64_t grid) {
    if (grid <= 0) return 0;
    const int n = a.S.n, R = a.S.m;
    int npad = 1;
    while (npad < n) npad <<= 1;
    a.npad = npad;
    a.order = order;
    const char *what = order > 0 ? "OSD-CS" : "OSD-0";
    int unused;
    const size_t smem = osd_smem(a, R, false, &unused);
    // FBGNN_OSD_CLUSTER=<C> (2, 4 or 8; read at every launch) runs the cluster kernel where one CTA would do, so that
    // small codes test it against k_osd.
    int force = 0;
    if (const char *e = getenv("FBGNN_OSD_CLUSTER")) {
        force = atoi(e);
        REQUIRE(force == 2 || force == 4 || force == 8, "FBGNN_OSD_CLUSTER=%s: expected 2, 4 or 8", e);
    }
    if (!force && smem <= ctx->smem_optin) {
        if (int rc = set_smem(k_osd, smem, ctx, what)) return rc;
        k_osd<<<(unsigned)grid, 256, smem, ctx->stream>>>(a);
        CK(cudaGetLastError());
        ctx->launches++;
        return 0;
    }
    // The matrix exceeds one CTA: the smallest cluster of 2 / 4 / 8 CTAs whose per-CTA rows fit (fbgnn_osd_cluster.cuh).
    // Every CTA gets the largest per-rank footprint: its share of the rows plus, for rank 0, the OSD-CS vectors.
    size_t smem_cl = 0;
    for (int C = force ? force : 2; C <= OSD_CL_MAX; C *= 2) {
        OsdCluster P{};
        P.C = C;
        P.rs = ((R + 31) / 32 + C - 1) / C * 32;
        smem_cl = osd_smem(a, P.rs, true, &P.slot_off);
        if (smem_cl > ctx->smem_optin) {
            if (force) break;
            continue;
        }
        CK(cudaFuncSetAttribute(k_osd_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cl));
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(grid * C), 1, 1);
        cfg.blockDim = dim3(256, 1, 1);
        cfg.dynamicSmemBytes = smem_cl;
        cfg.stream = ctx->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        int clusters = 0;
        CK(cudaOccupancyMaxActiveClusters(&clusters, k_osd_cluster, &cfg));
        if (clusters <= 0) {
            if (force) break;
            continue;
        }
        CK(cudaLaunchKernelEx(&cfg, k_osd_cluster, a, P));
        ctx->launches++;
        return 0;
    }
    return fail(FBGNN_E_UNSUPPORTED, "%s needs %zu bytes of shared memory per frame in one CTA and %zu per CTA in a "
                "cluster of %d; the device offers %zu per CTA", what, smem, smem_cl, force ? force : OSD_CL_MAX,
                ctx->smem_optin);
}

// OSD-CS candidate indices are 32-bit: 1 + N + lp (lp - 1) / 2 < 2^32 for lp <= 65535
static int check_osd_order(int32_t order) {
    REQUIRE(order >= 0 && order <= 65535, "OSD order %d outside [0, 65535]", order);
    return 0;
}

extern "C" int fbgnn_osd_decode(fbgnn_graph *basis, int32_t order, int64_t B, fbgnn_tensor2 llr, fbgnn_tensor2 synd,
                                fbgnn_tensor2 e_hat) {
    REQUIRE(basis && llr.ptr && synd.ptr && e_hat.ptr && B >= 0, "bad argument");
    if (int rc = check_osd_order(order)) return rc;
    if (int rc = need_decodable(basis)) return rc;
    fbgnn_ctx *ctx = basis->ctx;
    if (set_device(ctx)) return FBGNN_E_CUDA;
    OsdArgs a{};
    a.S = basis->dev;
    a.llr = v2<const float>(llr); a.sign = 1.0f;
    a.synd = v2<const uint8_t>(synd);
    a.e_hat = v2<uint8_t>(e_hat);
    return launch_osd(ctx, a, order, B);
}

extern "C" int fbgnn_osd0_decode(fbgnn_graph *basis, int64_t B, fbgnn_tensor2 llr, fbgnn_tensor2 synd,
                                 fbgnn_tensor2 e_hat) {
    return fbgnn_osd_decode(basis, 0, B, llr, synd, e_hat);
}

// ------------------------------------------------------------------ LSD-0 ---------------
// Budgets: 0 = the default; otherwise [1, limit].  The limits keep the worst case (n = m = 65535) inside one CTA.
static int lsd_budgets(int32_t *max_cols, int32_t *max_checks) {
    if (*max_cols == 0) *max_cols = LSD_DEF_COLS;
    if (*max_checks == 0) *max_checks = LSD_DEF_CHECKS;
    REQUIRE(*max_cols >= 1 && *max_cols <= LSD_MAX_COLS, "LSD max_cols %d outside [1, %d]", *max_cols, LSD_MAX_COLS);
    REQUIRE(*max_checks >= 1 && *max_checks <= LSD_MAX_CHECKS, "LSD max_checks %d outside [1, %d]", *max_checks,
            LSD_MAX_CHECKS);
    return 0;
}

static int launch_lsd(fbgnn_ctx *ctx, LsdArgs &a, int64_t grid) {
    if (grid <= 0) return 0;
    const size_t smem = LsdLayout(a.S.n, a.S.m, a.max_cols, a.max_checks).total;
    if (int rc = set_smem(k_lsd, smem, ctx, "LSD-0")) return rc;
    k_lsd<<<(unsigned)grid, 256, smem, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}

extern "C" int fbgnn_lsd_decode(fbgnn_graph *pcm, int32_t max_cols, int32_t max_checks, int64_t B, fbgnn_tensor2 llr,
                                fbgnn_tensor2 synd, fbgnn_tensor2 e_hat, uint8_t *status) {
    REQUIRE(pcm && llr.ptr && synd.ptr && B >= 0 && B < ((int64_t)1 << 31), "bad argument");
    if (int rc = lsd_budgets(&max_cols, &max_checks)) return rc;
    if (int rc = need_decodable(pcm)) return rc;
    fbgnn_ctx *ctx = pcm->ctx;
    if (set_device(ctx)) return FBGNN_E_CUDA;
    LsdArgs a{};
    a.S = pcm->dev;
    a.llr = v2<const float>(llr); a.sign = 1.0f;
    a.synd = v2<const uint8_t>(synd);
    a.e_hat = v2<uint8_t>(e_hat);
    a.status = status;
    a.max_cols = max_cols; a.max_checks = max_checks;
    return launch_lsd(ctx, a, B);
}

// ------------------------------------------------------------------ pipelines -----------
static int ws_reserve(fbgnn_ctx *ctx, int64_t B, int n, int m) {
    Workspace &w = ctx->ws;
    if (w.cap_frames >= B && w.n == n && w.m == m) return 0;
    CK(cudaStreamSynchronize(ctx->stream));
    ws_free(w);
    const size_t b = (size_t)B;
    CK(cudaMalloc(&w.vbits, b * n));
    CK(cudaMalloc(&w.sbits, b * (size_t)pad16(std::max(m, 1))));          // rows padded to 16 bytes (bulk-async staging)
    CK(cudaMalloc(&w.active[0], b));
    CK(cudaMalloc(&w.active[1], b));
    CK(cudaMalloc(&w.rounds, b));
    CK(cudaMalloc(&w.iters, b));
    CK(cudaMalloc(&w.L, b * 3 * n * sizeof(float)));
    CK(cudaMalloc(&w.P, b * 3 * (size_t)pad4(n) * sizeof(float)));        // [B][3][pad4(n)]: 16-byte aligned frame blocks
    CK(cudaMalloc(&w.logit, b * std::max(m, 1) * sizeof(float)));
    CK(cudaMalloc(&w.list[0], b * sizeof(int)));
    CK(cudaMalloc(&w.list[1], b * sizeof(int)));
    CK(cudaMalloc(&w.list_count, 2 * sizeof(int)));
    CK(cudaMalloc(&w.counters, 4 * sizeof(unsigned long long)));
    w.cap_frames = B; w.n = n; w.m = m;
    return 0;
}

struct PackedIO {                   // packed bit-plane variants of the pipeline's inputs / outputs (fbgnn_pipeline_run_bits)
    const uint32_t *nx_words = nullptr, *nz_words = nullptr;
    uint32_t *frame_bits = nullptr, *xd_words = nullptr, *zd_words = nullptr;
};

static int pipeline_run_impl(fbgnn_code *code, const fbgnn_pipeline_cfg *cfg, uint64_t seed,
                             uint64_t first_frame, int64_t B, fbgnn_tensor2 noise_x, fbgnn_tensor2 noise_z,
                             uint8_t *flags, fbgnn_tensor2 x_diff, fbgnn_tensor2 z_diff, int64_t *counters,
                             const PackedIO &pk);

extern "C" int fbgnn_pipeline_run(fbgnn_code *code, const fbgnn_pipeline_cfg *cfg, uint64_t seed,
                                  uint64_t first_frame, int64_t B, fbgnn_tensor2 noise_x, fbgnn_tensor2 noise_z,
                                  uint8_t *flags, fbgnn_tensor2 x_diff, fbgnn_tensor2 z_diff, int64_t *counters) {
    return pipeline_run_impl(code, cfg, seed, first_frame, B, noise_x, noise_z, flags, x_diff, z_diff, counters, PackedIO());
}

extern "C" int fbgnn_pipeline_run_bits(fbgnn_code *code, const fbgnn_pipeline_cfg *cfg, uint64_t seed,
                                       uint64_t first_frame, int64_t B, const uint32_t *noise_x_bits,
                                       const uint32_t *noise_z_bits, uint32_t *frame_bits, uint32_t *x_diff_bits,
                                       uint32_t *z_diff_bits, int64_t *counters) {
    REQUIRE((noise_x_bits == nullptr) == (noise_z_bits == nullptr), "give both noise planes or neither");
    PackedIO pk;
    pk.nx_words = noise_x_bits; pk.nz_words = noise_z_bits;
    pk.frame_bits = frame_bits; pk.xd_words = x_diff_bits; pk.zd_words = z_diff_bits;
    const fbgnn_tensor2 none = {nullptr, 0, 0};
    return pipeline_run_impl(code, cfg, seed, first_frame, B, none, none, nullptr, none, none, counters, pk);
}

static int pipeline_run_impl(fbgnn_code *code, const fbgnn_pipeline_cfg *cfg, uint64_t seed,
                             uint64_t first_frame, int64_t B, fbgnn_tensor2 noise_x, fbgnn_tensor2 noise_z,
                             uint8_t *flags, fbgnn_tensor2 x_diff, fbgnn_tensor2 z_diff, int64_t *counters,
                             const PackedIO &pk) {
    REQUIRE(code && cfg, "NULL argument");
    REQUIRE(cfg->num_stages >= 1 && cfg->num_iter && cfg->factor && cfg->cn_type, "bad pipeline configuration");
    REQUIRE(cfg->num_stages == 1 || cfg->gnn, "feedback GNNs missing");
    REQUIRE((noise_x.ptr == nullptr) == (noise_z.ptr == nullptr), "give both noise_x and noise_z or neither");
    REQUIRE(B >= 0 && B < ((int64_t)1 << 31), "bad batch size");
    REQUIRE(!cfg->osd0 || cfg->lsd || (code->basis_x && code->basis_z), "OSD-0 needs fbgnn_code_set_basis first");
    if (int rc = check_osd_order(cfg->osd_order)) return rc;
    int32_t lsd_cols = cfg->lsd_max_cols, lsd_checks = cfg->lsd_max_checks;
    if (cfg->osd0 && cfg->lsd)
        if (int rc = lsd_budgets(&lsd_cols, &lsd_checks)) return rc;
    REQUIRE(cfg->fixed_weight <= 0 || code->X->dev.n <= 65535, "fixed-weight sampling shuffles uint16 qubit indices (n <= 65535)");
    for (int s = 0; s < cfg->num_stages; s++) {
        REQUIRE(cfg->cn_type[s] >= 0 && cfg->cn_type[s] <= 2, "unknown cn_type in stage %d", s);
        REQUIRE(cfg->num_iter[s] >= 0, "negative num_iter in stage %d", s);
        REQUIRE(!cfg->early_stop || cfg->num_iter[s] <= 255, "early stop needs num_iter <= 255 (stage %d)", s);
        REQUIRE(s == 0 || cfg->gnn[s - 1], "feedback GNN %d is NULL", s - 1);
    }
    fbgnn_ctx *ctx = code->ctx;
    if (set_device(ctx)) return FBGNN_E_CUDA;
    const SideDev &X = code->X->dev, &Z = code->Z->dev;
    const int n = X.n, m = X.m + Z.m;
    if (counters) std::memset(counters, 0, 4 * sizeof(int64_t));
    if (B == 0) return 0;
    if (int rc = ws_reserve(ctx, B, n, m)) return rc;
    Workspace &w = ctx->ws;
    cudaStream_t st = ctx->stream;
    CK(cudaMemsetAsync(w.rounds, 0, (size_t)B, st));
    CK(cudaMemsetAsync(w.counters, 0, 4 * sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(w.list_count, 0, 2 * sizeof(int), st));

    // noise + syndromes
    SampleArgs sa{};
    sa.X = X; sa.Z = Z; sa.mode = cfg->fixed_weight > 0 ? 2 : 0; sa.wt = cfg->fixed_weight;
    sa.thr0 = cfg->thr[0]; sa.thr1 = cfg->thr[1]; sa.thr2 = cfg->thr[2];
    sa.seed = seed; sa.first_frame = first_frame;
    sa.nx_in = v2<const uint8_t>(noise_x); sa.nz_in = v2<const uint8_t>(noise_z);
    const int wq = pad4((n + 31) / 32);                  // words per packed qubit plane (rows 16-byte aligned)
    sa.nx_words = pk.nx_words; sa.nz_words = pk.nz_words; sa.wq = wq;
    const int np = pad4(n), mp = pad16(m);
    sa.vbits = w.vbits; sa.sbits = w.sbits; sa.sb_stride = mp;
    k_sample<<<(unsigned)B, 128, (size_t)3 * n + 8, st>>>(sa);
    CK(cudaGetLastError());
    ctx->launches++;

    const int S = cfg->num_stages;
    int64_t cur_count = B;            // frames the current stage runs on
    const int *cur_list = nullptr;
    for (int s = 0; s < S; s++) {
        const bool last = (s == S - 1);
        if (s > 0) {
            // feedbacks[s-1]: priors P from the marginals L and the soft syndromes
            GnnArgs ga{};
            ga.X = X; ga.Z = Z;
            ga.frame_list = cur_list; ga.num_frames = cur_count;
            ga.h_vn = View3<const float>{w.L, 3 * (int64_t)n, 1, n};
            ga.logit_hx = View2<const float>{w.logit, 1, m};           // z_logit: rows of hx
            ga.logit_hz = View2<const float>{w.logit + X.m, 1, m};     // x_logit: rows of hz
            ga.sx = View2<const uint8_t>{w.sbits, 1, mp};
            ga.sz = View2<const uint8_t>{w.sbits + X.m, 1, mp};
            ga.out = View3<float>{w.P, 3 * (int64_t)np, 1, np};
            if (int rc = launch_gnn(ctx, cfg->gnn[s - 1], ga)) return rc;
        }
        Bp4Args a{};
        a.X = X; a.Z = Z;
        a.cn_type = cfg->cn_type[s]; a.num_iter = cfg->num_iter[s]; a.factor = cfg->factor[s];
        a.frame_list = cur_list;
        if (s > 0) { a.llr = View3<const float>{w.P, 3 * (int64_t)np, np, 1}; a.llr_bulk = w.P; }
        a.prior = cfg->prior;
        a.sx = View2<const uint8_t>{w.sbits, 1, mp};
        a.sz = View2<const uint8_t>{w.sbits + X.m, 1, mp};
        a.synd_bulk = w.sbits;
        if (!last || cfg->osd0) {
            a.Lx = View2<float>{w.L, 3 * (int64_t)n, 1};
            a.Ly = View2<float>{w.L + n, 3 * (int64_t)n, 1};
            a.Lz = View2<float>{w.L + 2 * n, 3 * (int64_t)n, 1};
            if (!last) {
                a.zl = View2<float>{w.logit, 1, m};
                a.xl = View2<float>{w.logit + X.m, 1, m};
            }
        }
        a.vbits = w.vbits;
        a.iters_out = cfg->early_stop ? w.iters : nullptr;
        a.active_in = (s == 0) ? nullptr : w.active[(s - 1) & 1];
        a.active_out = w.active[s & 1];
        a.rounds = last ? nullptr : w.rounds;
        const bool compact = (cfg->skip_inactive && !last) || (last && cfg->osd0);
        if (compact) {
            CK(cudaMemsetAsync(w.list_count + (s & 1), 0, sizeof(int), st));
            a.next_list = w.list[s & 1];
            a.next_count = w.list_count + (s & 1);
        }
        if (int rc = launch_bp4(ctx, a, cur_count)) return rc;
        if (compact) {
            int cnt = 0;
            CK(cudaMemcpyAsync(&cnt, w.list_count + (s & 1), sizeof(int), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            cur_count = cnt;
            cur_list = w.list[s & 1];
            if (cur_count == 0) break;
        }
    }

    if (cfg->osd0 && cur_count > 0 && cur_list) {
        // BP4_OSD_Model (bp_osd.py:80-197): frames still mismatching get both parts re-solved by OSD-0
        OsdLlrArgs la{n, cur_list, cur_count, w.L, w.P, np};
        const int64_t blocks = std::min<int64_t>((cur_count * n + 255) / 256, (int64_t)ctx->num_sms * 8);
        if (ctx->math_mode == FBGNN_MATH_SFU) k_osd_llr<MathSfu><<<(unsigned)blocks, 256, 0, st>>>(la);
        else k_osd_llr<MathExact><<<(unsigned)blocks, 256, 0, st>>>(la);
        CK(cudaGetLastError());
        ctx->launches++;
        if (cfg->lsd) {
            // LSD-0 on each side's full matrix; a side it abandons keeps its BP decision
            LsdArgs ls{};
            ls.frame_list = cur_list; ls.sign = 1.0f;
            ls.vbits = w.vbits;
            ls.max_cols = lsd_cols; ls.max_checks = lsd_checks;
            ls.S = X;                                                    // hx, osd_llrz, syndrome_x -> z_hat
            ls.llr = View2<const float>{w.P + np, 3 * (int64_t)np, 1};
            ls.synd = View2<const uint8_t>{w.sbits, 1, mp}; ls.vbit = 3;
            if (int rc = launch_lsd(ctx, ls, cur_count)) return rc;
            ls.S = Z;                                                    // hz, osd_llrx, syndrome_z -> x_hat
            ls.llr = View2<const float>{w.P, 3 * (int64_t)np, 1};
            ls.synd = View2<const uint8_t>{w.sbits + X.m, 1, mp}; ls.vbit = 2;
            if (int rc = launch_lsd(ctx, ls, cur_count)) return rc;
        } else {
        OsdArgs oa{};
        oa.frame_list = cur_list; oa.sign = 1.0f;
        oa.vbits = w.vbits;
        oa.S = code->basis_x->dev;                                   // hx basis, osd_llrz, syndrome_x -> z_hat
        oa.llr = View2<const float>{w.P + np, 3 * (int64_t)np, 1};
        oa.synd = View2<const uint8_t>{w.sbits, 1, mp}; oa.synd_row = code->pivot_x; oa.vbit = 3;
        if (int rc = launch_osd(ctx, oa, cfg->osd_order, cur_count)) return rc;
        oa.S = code->basis_z->dev;                                   // hz basis, osd_llrx, syndrome_z -> x_hat
        oa.llr = View2<const float>{w.P, 3 * (int64_t)np, 1};
        oa.synd = View2<const uint8_t>{w.sbits + X.m, 1, mp}; oa.synd_row = code->pivot_z; oa.vbit = 2;
        if (int rc = launch_osd(ctx, oa, cfg->osd_order, cur_count)) return rc;
        }
    }

    FinalArgs fa{};
    fa.X = X; fa.Z = Z;
    fa.lx_bits = code->lx_bits; fa.lz_bits = code->lz_bits; fa.kx = code->kx; fa.kz = code->kz;
    fa.binary = 0;
    fa.vbits = w.vbits; fa.rounds = w.rounds; fa.flags = flags;
    fa.x_diff = v2<uint8_t>(x_diff); fa.z_diff = v2<uint8_t>(z_diff);
    fa.counters = w.counters;
    if (pk.frame_bits) {
        fa.frame_bits = pk.frame_bits; fa.fw = (B + 31) / 32;
        CK(cudaMemsetAsync(pk.frame_bits, 0, sizeof(uint32_t) * 3 * (size_t)fa.fw, st));
    }
    fa.xd_words = pk.xd_words; fa.zd_words = pk.zd_words; fa.wq = wq;
    const int W = (n + 31) / 32;
    k_final<<<(unsigned)B, 128, (size_t)((n + 3) & ~3) + 8 * (size_t)W, st>>>(fa);
    CK(cudaGetLastError());
    ctx->launches++;
    if (counters) {
        unsigned long long h[4];
        CK(cudaMemcpyAsync(h, w.counters, sizeof h, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (int i = 0; i < 4; i++) counters[i] = (int64_t)h[i];
    }
    return 0;
}

extern "C" int fbgnn_bsc_pipeline_run(fbgnn_graph *g, fbgnn_graph *logical, int32_t cn_type, int32_t num_iter,
                                      float factor, float llr_const, float p, uint64_t seed, uint64_t first_frame,
                                      int64_t B, fbgnn_tensor2 noise, uint8_t *flags, int64_t *counters,
                                      fbgnn_graph *osd_basis, const int32_t *osd_pivot) {
    return fbgnn_bsc_pipeline_run_ex(g, logical, cn_type, num_iter, factor, llr_const, p, seed, first_frame, B, noise,
                                     flags, counters, osd_basis, osd_pivot, 0);
}

// BP_BSC_Model with, on the frames BP2 leaves mismatching, OSD on osd_basis or (lsd) LSD-0 on g itself
static int bsc_pipeline_impl(fbgnn_graph *g, fbgnn_graph *logical, int32_t cn_type, int32_t num_iter, float factor,
                             float llr_const, float p, uint64_t seed, uint64_t first_frame, int64_t B,
                             fbgnn_tensor2 noise, uint8_t *flags, int64_t *counters, fbgnn_graph *osd_basis,
                             const int32_t *osd_pivot, int32_t osd_order, bool lsd, int32_t lsd_cols,
                             int32_t lsd_checks) {
    REQUIRE(g, "graph is NULL");
    if (lsd)
        if (int rc = lsd_budgets(&lsd_cols, &lsd_checks)) return rc;
    if (int rc = check_osd_order(osd_order)) return rc;
    REQUIRE(!osd_basis || (osd_pivot && osd_basis->dev.n == g->dev.n && osd_basis->dev.m <= g->dev.m),
            "bad OSD-0 basis");
    REQUIRE(cn_type >= 0 && cn_type <= 2, "unknown cn_type %d", cn_type);
    REQUIRE(num_iter >= 0 && B >= 0 && B < ((int64_t)1 << 31), "bad argument");
    REQUIRE(!logical || logical->dev.n == g->dev.n, "logical_pcm has %d columns, pcm has %d",
            logical ? logical->dev.n : 0, g->dev.n);
    if (int rc = need_decodable(g)) return rc;
    fbgnn_ctx *ctx = g->ctx;
    if (set_device(ctx)) return FBGNN_E_CUDA;
    const SideDev &S = g->dev;
    const int n = S.n, m = S.m;
    if (counters) std::memset(counters, 0, 4 * sizeof(int64_t));
    if (B == 0) return 0;
    if (int rc = ws_reserve(ctx, B, n, m)) return rc;
    Workspace &w = ctx->ws;
    cudaStream_t st = ctx->stream;
    CK(cudaMemsetAsync(w.counters, 0, 4 * sizeof(unsigned long long), st));
    SampleArgs sa{};
    sa.X = S; sa.mode = 1; sa.thr0 = p;
    sa.seed = seed; sa.first_frame = first_frame;
    sa.nx_in = v2<const uint8_t>(noise);
    const int mp = pad16(m);
    sa.vbits = w.vbits; sa.sbits = w.sbits; sa.sb_stride = mp;
    k_sample<<<(unsigned)B, 128, (size_t)n, st>>>(sa);
    CK(cudaGetLastError());
    ctx->launches++;
    Bp2Args a{};
    a.S = S; a.cn_type = cn_type; a.num_iter = num_iter; a.factor = factor;
    a.llr_const = llr_const;
    a.synd = View2<const uint8_t>{w.sbits, 1, mp};
    a.vbits = w.vbits;                 // decision -> bit 2
    if (osd_basis || lsd) {
        CK(cudaMemsetAsync(w.list_count, 0, sizeof(int), st));
        a.soft = View2<float>{w.L, n, 1};
        a.next_list = w.list[0]; a.next_count = w.list_count;
    }
    if (int rc = launch_bp2(ctx, a, B)) return rc;
    if (lsd) {
        int cnt = 0;
        CK(cudaMemcpyAsync(&cnt, w.list_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        LsdArgs ls{};
        ls.S = S; ls.frame_list = w.list[0];
        ls.llr = View2<const float>{w.L, n, 1}; ls.sign = -1.0f;         // llr_hat = -decoder output
        ls.synd = View2<const uint8_t>{w.sbits, 1, mp};
        ls.vbits = w.vbits; ls.vbit = 2;
        ls.max_cols = lsd_cols; ls.max_checks = lsd_checks;
        if (int rc = launch_lsd(ctx, ls, cnt)) return rc;
    } else if (osd_basis) {
        // BP2_OSD_Model (bp_osd.py:199-274): OSD-0 on the frames whose decision misses the syndrome
        if (int rc = need_decodable(osd_basis)) return rc;
        int cnt = 0;
        CK(cudaMemcpyAsync(&cnt, w.list_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (cnt > 0) {
            const int R = osd_basis->dev.m;
            std::vector<idx_t> piv(R);
            for (int r = 0; r < R; r++) {
                REQUIRE(osd_pivot[r] >= 0 && osd_pivot[r] < m, "pivot row out of range");
                piv[r] = (idx_t)osd_pivot[r];
            }
            idx_t *dp = nullptr;
            CK(cudaMallocAsync(&dp, R * sizeof(idx_t), st));
            CK(cudaMemcpyAsync(dp, piv.data(), R * sizeof(idx_t), cudaMemcpyHostToDevice, st));
            OsdArgs oa{};
            oa.S = osd_basis->dev; oa.frame_list = w.list[0];
            oa.llr = View2<const float>{w.L, n, 1}; oa.sign = -1.0f;      // llr_hat = -decoder output
            oa.synd = View2<const uint8_t>{w.sbits, 1, mp}; oa.synd_row = dp;
            oa.vbits = w.vbits; oa.vbit = 2;
            if (int rc = launch_osd(ctx, oa, osd_order, cnt)) return rc;
            CK(cudaStreamSynchronize(st));                                  // piv must outlive the copy
            CK(cudaFreeAsync(dp, st));
        }
    }
    FinalArgs fa{};
    fa.X = S;
    fa.lx_bits = logical ? logical->dev.bitrows : nullptr;
    fa.kx = logical ? logical->dev.m : 0;
    fa.binary = 1;
    fa.vbits = w.vbits; fa.flags = flags; fa.counters = w.counters;
    const int W = (n + 31) / 32;
    k_final<<<(unsigned)B, 128, (size_t)((n + 3) & ~3) + 8 * (size_t)W, st>>>(fa);
    CK(cudaGetLastError());
    ctx->launches++;
    if (counters) {
        unsigned long long h[4];
        CK(cudaMemcpyAsync(h, w.counters, sizeof h, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (int i = 0; i < 4; i++) counters[i] = (int64_t)h[i];
    }
    return 0;
}

extern "C" int fbgnn_bsc_pipeline_run_ex(fbgnn_graph *g, fbgnn_graph *logical, int32_t cn_type, int32_t num_iter,
                                         float factor, float llr_const, float p, uint64_t seed, uint64_t first_frame,
                                         int64_t B, fbgnn_tensor2 noise, uint8_t *flags, int64_t *counters,
                                         fbgnn_graph *osd_basis, const int32_t *osd_pivot, int32_t osd_order) {
    return bsc_pipeline_impl(g, logical, cn_type, num_iter, factor, llr_const, p, seed, first_frame, B, noise, flags,
                             counters, osd_basis, osd_pivot, osd_order, false, 0, 0);
}

extern "C" int fbgnn_bsc_pipeline_run_lsd(fbgnn_graph *g, fbgnn_graph *logical, int32_t cn_type, int32_t num_iter,
                                          float factor, float llr_const, float p, uint64_t seed, uint64_t first_frame,
                                          int64_t B, fbgnn_tensor2 noise, uint8_t *flags, int64_t *counters,
                                          int32_t max_cols, int32_t max_checks) {
    return bsc_pipeline_impl(g, logical, cn_type, num_iter, factor, llr_const, p, seed, first_frame, B, noise, flags,
                             counters, nullptr, nullptr, 0, true, max_cols, max_checks);
}
