// fbgnn_core.cu -- C ABI (include/fbgnn.h): library / context / memory / graph handles, noise sources,
// measurement probes.  No CPU compute path: every entry point that does work launches CUDA kernels and
// fails with FBGNN_E_CUDA when there is no device.
#include "fbgnn_internal.h"

// ------------------------------------------------------------------ errors -------------
static thread_local std::string g_err;

int fbgnn_fail(int code, const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

// ------------------------------------------------------------------ library / context ---
extern "C" int fbgnn_version(void) { return FBGNN_VERSION; }
extern "C" const char *fbgnn_last_error(void) { return g_err.c_str(); }

extern "C" int fbgnn_device_count(int *count) {
    REQUIRE(count, "count is NULL");
    CK(cudaGetDeviceCount(count));
    return 0;
}

extern "C" int fbgnn_ctx_create(int device, fbgnn_ctx **out) {
    REQUIRE(out, "ctx is NULL");
    int count = 0;
    CK(cudaGetDeviceCount(&count));
    REQUIRE(device >= 0 && device < count, "device %d out of range (%d devices)", device, count);
    CK(cudaSetDevice(device));
    fbgnn_ctx *ctx = new fbgnn_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    ctx->num_sms = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    snprintf(ctx->name, sizeof ctx->name, "%s", prop.name);
    CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    {
        cudaMemPool_t pool;
        CK(cudaDeviceGetDefaultMemPool(&pool, device));
        uint64_t keep = UINT64_MAX;
        CK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    CK(cudaEventCreate(&ctx->ev0));
    CK(cudaEventCreate(&ctx->ev1));
    *out = ctx;
    return 0;
}

void ws_free(Workspace &w) {
    cudaFree(w.vbits); cudaFree(w.sbits); cudaFree(w.active[0]); cudaFree(w.active[1]);
    cudaFree(w.rounds); cudaFree(w.iters); cudaFree(w.L); cudaFree(w.P); cudaFree(w.logit); cudaFree(w.list[0]);
    cudaFree(w.list[1]); cudaFree(w.list_count); cudaFree(w.counters);
    w = Workspace();
}

extern "C" int fbgnn_ctx_destroy(fbgnn_ctx *ctx) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    fbgnn_comm_destroy(ctx);
    cudaFree(ctx->comm_buf);
    cudaFree(ctx->stats);
    ws_free(ctx->ws);
    cudaFree(ctx->flush_buf);
    cudaEventDestroy(ctx->ev0);
    cudaEventDestroy(ctx->ev1);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return 0;
}

extern "C" int fbgnn_ctx_sync(fbgnn_ctx *ctx) {
    REQUIRE(ctx, "ctx is NULL");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int fbgnn_ctx_device(fbgnn_ctx *ctx, int *device, int *num_sms, char *name, int name_len) {
    REQUIRE(ctx, "ctx is NULL");
    if (device) *device = ctx->device;
    if (num_sms) *num_sms = ctx->num_sms;
    if (name && name_len > 0) snprintf(name, (size_t)name_len, "%s", ctx->name);
    return 0;
}

extern "C" int fbgnn_timer_start(fbgnn_ctx *ctx) {
    REQUIRE(ctx, "ctx is NULL");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    return 0;
}

extern "C" int fbgnn_timer_stop(fbgnn_ctx *ctx, float *ms) {
    REQUIRE(ctx && ms, "NULL argument");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaEventSynchronize(ctx->ev1));
    CK(cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
    return 0;
}

extern "C" int fbgnn_ctx_set_math(fbgnn_ctx *ctx, int32_t mode) {
    REQUIRE(ctx, "ctx is NULL");
    REQUIRE(mode == FBGNN_MATH_EXACT || mode == FBGNN_MATH_SFU, "unknown math mode %d", mode);
    ctx->math_mode = mode;
    return 0;
}

extern "C" int fbgnn_ctx_get_math(fbgnn_ctx *ctx, int32_t *mode) {
    REQUIRE(ctx && mode, "NULL argument");
    *mode = ctx->math_mode;
    return 0;
}

extern "C" int fbgnn_ctx_stats(fbgnn_ctx *ctx, int64_t out[2], int32_t reset) {
    REQUIRE(ctx, "ctx is NULL");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    if (!ctx->stats) {
        CK(cudaMalloc(&ctx->stats, 2 * sizeof(unsigned long long)));
        CK(cudaMemsetAsync(ctx->stats, 0, 2 * sizeof(unsigned long long), ctx->stream));
    }
    if (out) {
        unsigned long long h[2];
        CK(cudaMemcpyAsync(h, ctx->stats, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        out[0] = (int64_t)h[0]; out[1] = (int64_t)h[1];
    }
    if (reset) CK(cudaMemsetAsync(ctx->stats, 0, 2 * sizeof(unsigned long long), ctx->stream));
    return 0;
}

extern "C" int fbgnn_launch_count(fbgnn_ctx *ctx, int64_t *launches) {
    REQUIRE(ctx && launches, "NULL argument");
    *launches = ctx->launches;
    return 0;
}

// ------------------------------------------------------------------ memory --------------
// Stream-ordered allocation from the device's default memory pool (kept cached: the release
// threshold is raised at context creation), so per-call output tensors cost no cudaMalloc.
extern "C" int fbgnn_malloc(fbgnn_ctx *ctx, size_t bytes, void **dptr) {
    REQUIRE(ctx && dptr, "NULL argument");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    cudaError_t e = cudaMallocAsync(dptr, bytes ? bytes : 1, ctx->stream);
    if (e == cudaErrorMemoryAllocation) { cudaGetLastError(); return fail(FBGNN_E_NOMEM, "cudaMallocAsync(%zu) out of memory", bytes); }
    CK(e);
    return 0;
}
extern "C" int fbgnn_free(fbgnn_ctx *ctx, void *dptr) {
    REQUIRE(ctx, "ctx is NULL");
    if (!dptr) return 0;
    if (set_device(ctx)) return FBGNN_E_CUDA;
    CK(cudaFreeAsync(dptr, ctx->stream));
    return 0;
}
extern "C" int fbgnn_memset(fbgnn_ctx *ctx, void *dptr, int value, size_t bytes) {
    REQUIRE(ctx, "ctx is NULL");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    CK(cudaMemsetAsync(dptr, value, bytes, ctx->stream));
    return 0;
}
extern "C" int fbgnn_memcpy_h2d(fbgnn_ctx *ctx, void *dst, const void *src, size_t bytes) {
    REQUIRE(ctx, "ctx is NULL");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return 0;
}
extern "C" int fbgnn_memcpy_d2h(fbgnn_ctx *ctx, void *dst, const void *src, size_t bytes) {
    REQUIRE(ctx, "ctx is NULL");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}
extern "C" int fbgnn_memcpy_d2d(fbgnn_ctx *ctx, void *dst, const void *src, size_t bytes) {
    REQUIRE(ctx, "ctx is NULL");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return 0;
}
extern "C" int fbgnn_host_alloc(size_t bytes, void **hptr) {
    REQUIRE(hptr, "hptr is NULL");
    CK(cudaMallocHost(hptr, bytes ? bytes : 1));
    return 0;
}
extern "C" int fbgnn_host_free(void *hptr) {
    CK(cudaFreeHost(hptr));
    return 0;
}
extern "C" int fbgnn_flush_l2(fbgnn_ctx *ctx) {
    REQUIRE(ctx, "ctx is NULL");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    if (!ctx->flush_buf) {
        ctx->flush_bytes = (size_t)256 << 20;        // 256 MiB > 126 MB of L2
        CK(cudaMalloc(&ctx->flush_buf, ctx->flush_bytes));
    }
    k_fill<<<ctx->num_sms * 4, 256, 0, ctx->stream>>>((uint32_t *)ctx->flush_buf,
                                                      (int64_t)(ctx->flush_bytes / 4), 0u);
    CK(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------ graphs --------------
template <typename T>
static int upload(fbgnn_graph *g, const std::vector<T> &h, const T **dptr) {
    void *d = nullptr;
    CK(cudaMalloc(&d, std::max<size_t>(h.size(), 1) * sizeof(T)));
    g->allocs.push_back(d);
    if (!h.empty()) CK(cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    *dptr = (const T *)d;
    return 0;
}

static void pack_rows(int32_t n, int32_t m, const int32_t *indptr, const int32_t *indices,
                      std::vector<uint32_t> &bits) {
    const int W = (n + 31) / 32;
    bits.assign((size_t)std::max(m, 0) * W, 0u);
    for (int r = 0; r < m; r++)
        for (int k = indptr[r]; k < indptr[r + 1]; k++)
            bits[(size_t)r * W + (indices[k] >> 5)] ^= 1u << (indices[k] & 31);
}

static int validate_csr(int32_t n, int32_t m, const int32_t *indptr, const int32_t *indices, const char *what) {
    REQUIRE(n > 0 && m >= 0, "%s: bad shape (%d x %d)", what, m, n);
    REQUIRE(indptr && (indices || indptr[m] == 0), "%s: NULL CSR arrays", what);
    REQUIRE(indptr[0] == 0, "%s: indptr[0] != 0", what);
    for (int r = 0; r < m; r++) {
        REQUIRE(indptr[r + 1] >= indptr[r], "%s: indptr not monotone at row %d", what, r);
        for (int k = indptr[r]; k < indptr[r + 1]; k++) {
            REQUIRE(indices[k] >= 0 && indices[k] < n, "%s: column index %d out of range in row %d", what, indices[k], r);
            REQUIRE(k == indptr[r] || indices[k] > indices[k - 1], "%s: row %d not strictly increasing", what, r);
        }
    }
    return 0;
}

extern "C" int fbgnn_graph_create(fbgnn_ctx *ctx, int32_t n, int32_t m, const int32_t *indptr,
                                  const int32_t *indices, fbgnn_graph **out) {
    REQUIRE(ctx && out, "NULL argument");
    if (int rc = validate_csr(n, m, indptr, indices, "graph")) return rc;
    if (set_device(ctx)) return FBGNN_E_CUDA;
    const int E = indptr[m];
    fbgnn_graph *g = new fbgnn_graph();
    g->ctx = ctx;
    int max_dc = 0, max_dv = 0, min_dc = 1 << 30, min_dv = 1 << 30;
    for (int c = 0; c < m; c++) {
        const int dc = indptr[c + 1] - indptr[c];
        max_dc = std::max(max_dc, dc); min_dc = std::min(min_dc, dc);
    }
    char why[256] = {0};
    if (n > 65535 || m > 65535 || E > 65535)
        snprintf(why, sizeof why, "matrix too large for the shared-memory resident decoder (n=%d m=%d edges=%d; "
                 "limit 65535 each)", n, m, E);
    else if (max_dc > 64)
        snprintf(why, sizeof why, "check degree %d > 64 is not supported by the decoder", max_dc);
    g->decodable = why[0] == 0;
    g->why_not = why;
    // CN order is the CSR order (sorted by (cn, vn)); VN order = stable counting sort by vn.
    std::vector<idx_t> cn_ptr, cn_vn, cn_edge, vn_ptr, vn_cn;
    if (g->decodable) {
        cn_ptr.resize(m + 1); cn_vn.resize(E); cn_edge.resize(E); vn_ptr.resize(n + 1); vn_cn.resize(E);
        std::vector<int> deg(n, 0), fill(n, 0);
        for (int k = 0; k < E; k++) deg[indices[k]]++;
        int acc = 0;
        for (int v = 0; v < n; v++) { vn_ptr[v] = (idx_t)acc; fill[v] = acc; acc += deg[v]; }
        vn_ptr[n] = (idx_t)acc;
        for (int c = 0; c < m; c++) {
            cn_ptr[c] = (idx_t)indptr[c];
            for (int k = indptr[c]; k < indptr[c + 1]; k++) {
                const int v = indices[k];
                const int pos = fill[v]++;
                cn_vn[k] = (idx_t)v;
                cn_edge[k] = (idx_t)pos;
                vn_cn[pos] = (idx_t)c;
            }
        }
        cn_ptr[m] = (idx_t)E;
        for (int v = 0; v < n; v++) { max_dv = std::max(max_dv, deg[v]); min_dv = std::min(min_dv, deg[v]); }
    }
    g->max_dc = max_dc; g->max_dv = max_dv;
    std::vector<uint32_t> bits;
    pack_rows(n, m, indptr, indices, bits);
    SideDev &d = g->dev;
    d.n = n; d.m = m; d.E = E;
    d.reg_dc = (m > 0 && max_dc == min_dc) ? max_dc : 0;
    d.reg_dv = (max_dv == min_dv) ? max_dv : 0;
    g->h_vn_ptr.assign(vn_ptr.begin(), vn_ptr.end());
    d.h_vn_ptr = g->h_vn_ptr.empty() ? nullptr : g->h_vn_ptr.data();
    int rc = 0;
    rc |= upload(g, vn_ptr, &d.vn_ptr); rc |= upload(g, vn_cn, &d.vn_cn);
    rc |= upload(g, cn_ptr, &d.cn_ptr); rc |= upload(g, cn_edge, &d.cn_edge);
    rc |= upload(g, cn_vn, &d.cn_vn);   rc |= upload(g, bits, &d.bitrows);
    if (rc) { fbgnn_graph_destroy(g); return FBGNN_E_CUDA; }
    *out = g;
    return 0;
}

extern "C" int fbgnn_graph_destroy(fbgnn_graph *g) {
    if (!g) return 0;
    cudaSetDevice(g->ctx->device);
    for (void *p : g->allocs) cudaFree(p);
    delete g;
    return 0;
}

extern "C" int fbgnn_code_create(fbgnn_ctx *ctx, int32_t n, int32_t m_x, const int32_t *hx_indptr,
                                 const int32_t *hx_indices, int32_t m_z, const int32_t *hz_indptr,
                                 const int32_t *hz_indices, int32_t k_x, const int32_t *lx_indptr,
                                 const int32_t *lx_indices, int32_t k_z, const int32_t *lz_indptr,
                                 const int32_t *lz_indices, fbgnn_code **out) {
    REQUIRE(ctx && out, "NULL argument");
    fbgnn_code *c = new fbgnn_code();
    c->ctx = ctx;
    c->X = c->Z = nullptr;
    int rc = fbgnn_graph_create(ctx, n, m_x, hx_indptr, hx_indices, &c->X);
    if (!rc) rc = fbgnn_graph_create(ctx, n, m_z, hz_indptr, hz_indices, &c->Z);
    if (!rc) rc = need_decodable(c->X);
    if (!rc) rc = need_decodable(c->Z);
    if (!rc && k_x > 0) rc = validate_csr(n, k_x, lx_indptr, lx_indices, "lx");
    if (!rc && k_z > 0) rc = validate_csr(n, k_z, lz_indptr, lz_indices, "lz");
    if (rc) { fbgnn_code_destroy(c); return rc; }
    c->kx = std::max(k_x, 0); c->kz = std::max(k_z, 0); c->W = (n + 31) / 32;
    c->hx_ptr.assign(hx_indptr, hx_indptr + m_x + 1); c->hx_idx.assign(hx_indices, hx_indices + hx_indptr[m_x]);
    c->hz_ptr.assign(hz_indptr, hz_indptr + m_z + 1); c->hz_idx.assign(hz_indices, hz_indices + hz_indptr[m_z]);
    std::vector<uint32_t> bits;
    auto up_rows = [&](int k, const int32_t *ptr, const int32_t *idx, int **dptr, idx_t **dcol) -> int {
        std::vector<int> p(ptr, ptr + k + 1);
        std::vector<idx_t> col(std::max(ptr[k], 1));
        for (int i = 0; i < ptr[k]; i++) col[i] = (idx_t)idx[i];
        CK(cudaMalloc(dptr, p.size() * sizeof(int)));
        CK(cudaMemcpy(*dptr, p.data(), p.size() * sizeof(int), cudaMemcpyHostToDevice));
        CK(cudaMalloc(dcol, col.size() * sizeof(idx_t)));
        CK(cudaMemcpy(*dcol, col.data(), col.size() * sizeof(idx_t), cudaMemcpyHostToDevice));
        return 0;
    };
    if (c->kx) if (int rc2 = up_rows(c->kx, lx_indptr, lx_indices, &c->lx_ptr, &c->lx_col)) return rc2;
    if (c->kz) if (int rc2 = up_rows(c->kz, lz_indptr, lz_indices, &c->lz_ptr, &c->lz_col)) return rc2;
    if (c->kx) {
        pack_rows(n, c->kx, lx_indptr, lx_indices, bits);
        CK(cudaMalloc(&c->lx_bits, bits.size() * 4));
        CK(cudaMemcpy(c->lx_bits, bits.data(), bits.size() * 4, cudaMemcpyHostToDevice));
    }
    if (c->kz) {
        pack_rows(n, c->kz, lz_indptr, lz_indices, bits);
        CK(cudaMalloc(&c->lz_bits, bits.size() * 4));
        CK(cudaMemcpy(c->lz_bits, bits.data(), bits.size() * 4, cudaMemcpyHostToDevice));
    }
    *out = c;
    return 0;
}

extern "C" int fbgnn_code_destroy(fbgnn_code *c) {
    if (!c) return 0;
    cudaSetDevice(c->ctx->device);
    fbgnn_graph_destroy(c->X);
    fbgnn_graph_destroy(c->Z);
    fbgnn_graph_destroy(c->basis_x);
    fbgnn_graph_destroy(c->basis_z);
    cudaFree(c->pivot_x);
    cudaFree(c->pivot_z);
    cudaFree(c->lx_ptr); cudaFree(c->lx_col); cudaFree(c->lz_ptr); cudaFree(c->lz_col);
    cudaFree(c->lx_bits);
    cudaFree(c->lz_bits);
    delete c;
    return 0;
}

static int make_basis(fbgnn_ctx *ctx, int n, const std::vector<int32_t> &ptr, const std::vector<int32_t> &idx,
                      int32_t rank, const int32_t *pivot, fbgnn_graph **graph, idx_t **dpivot) {
    const int m = (int)ptr.size() - 1;
    std::vector<int32_t> bp(1, 0), bi;
    std::vector<idx_t> piv(std::max(rank, 1));
    for (int r = 0; r < rank; r++) {
        REQUIRE(pivot[r] >= 0 && pivot[r] < m, "pivot row %d out of range", pivot[r]);
        bi.insert(bi.end(), idx.begin() + ptr[pivot[r]], idx.begin() + ptr[pivot[r] + 1]);
        bp.push_back((int32_t)bi.size());
        piv[r] = (idx_t)pivot[r];
    }
    if (int rc = fbgnn_graph_create(ctx, n, rank, bp.data(), bi.data(), graph)) return rc;
    CK(cudaMalloc(dpivot, piv.size() * sizeof(idx_t)));
    CK(cudaMemcpy(*dpivot, piv.data(), piv.size() * sizeof(idx_t), cudaMemcpyHostToDevice));
    return 0;
}

extern "C" int fbgnn_code_set_basis(fbgnn_code *code, int32_t rank_x, const int32_t *pivot_hx, int32_t rank_z,
                                    const int32_t *pivot_hz) {
    REQUIRE(code && pivot_hx && pivot_hz && rank_x > 0 && rank_z > 0, "bad argument");
    if (set_device(code->ctx)) return FBGNN_E_CUDA;
    fbgnn_graph_destroy(code->basis_x); code->basis_x = nullptr;
    fbgnn_graph_destroy(code->basis_z); code->basis_z = nullptr;
    cudaFree(code->pivot_x); code->pivot_x = nullptr;
    cudaFree(code->pivot_z); code->pivot_z = nullptr;
    const int n = code->X->dev.n;
    if (int rc = make_basis(code->ctx, n, code->hx_ptr, code->hx_idx, rank_x, pivot_hx, &code->basis_x, &code->pivot_x)) return rc;
    if (int rc = make_basis(code->ctx, n, code->hz_ptr, code->hz_idx, rank_z, pivot_hz, &code->basis_z, &code->pivot_z)) return rc;
    return 0;
}

extern "C" int fbgnn_code_edges(fbgnn_code *code, int32_t *e_x, int32_t *e_z) {
    REQUIRE(code, "code is NULL");
    if (e_x) *e_x = code->X->dev.E;
    if (e_z) *e_z = code->Z->dev.E;
    return 0;
}

// ------------------------------------------------------------------ noise sources -------
extern "C" int fbgnn_pauli_sample(fbgnn_ctx *ctx, int32_t n, int64_t B, const float thr[3], uint64_t seed,
                                  uint64_t first_frame, fbgnn_tensor2 noise_x, fbgnn_tensor2 noise_z) {
    REQUIRE(ctx && thr && n > 0 && B >= 0, "bad argument");
    REQUIRE(noise_x.ptr && noise_z.ptr, "noise outputs are NULL");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    if (B == 0) return 0;
    SampleArgs a{};
    a.X.n = n; a.mode = 0;
    a.thr0 = thr[0]; a.thr1 = thr[1]; a.thr2 = thr[2];
    a.seed = seed; a.first_frame = first_frame;
    a.nx_out = v2<uint8_t>(noise_x); a.nz_out = v2<uint8_t>(noise_z);
    k_sample<<<(unsigned)B, 128, (size_t)n, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}

extern "C" int fbgnn_pauli_sample_wt(fbgnn_ctx *ctx, int32_t n, int64_t B, int32_t wt, uint64_t seed,
                                     uint64_t first_frame, fbgnn_tensor2 noise_x, fbgnn_tensor2 noise_z) {
    REQUIRE(ctx && n > 0 && n <= 65535 && B >= 0 && wt >= 0, "bad argument");
    REQUIRE(noise_x.ptr && noise_z.ptr, "noise outputs are NULL");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    if (B == 0) return 0;
    SampleArgs a{};
    a.X.n = n; a.mode = 2; a.wt = wt;
    a.seed = seed; a.first_frame = first_frame;
    a.nx_out = v2<uint8_t>(noise_x); a.nz_out = v2<uint8_t>(noise_z);
    k_sample<<<(unsigned)B, 128, (size_t)3 * n + 8, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}

extern "C" int fbgnn_bsc_sample(fbgnn_ctx *ctx, int32_t n, int64_t B, float p, uint64_t seed,
                                uint64_t first_frame, fbgnn_tensor2 noise) {
    REQUIRE(ctx && n > 0 && B >= 0 && noise.ptr, "bad argument");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    if (B == 0) return 0;
    SampleArgs a{};
    a.X.n = n; a.mode = 1; a.thr0 = p;
    a.seed = seed; a.first_frame = first_frame;
    a.nx_out = v2<uint8_t>(noise);
    k_sample<<<(unsigned)B, 128, (size_t)n, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}

extern "C" int fbgnn_syndrome(fbgnn_graph *g, int64_t B, fbgnn_tensor2 noise, fbgnn_tensor2 syndrome) {
    REQUIRE(g && noise.ptr && syndrome.ptr && B >= 0, "bad argument");
    if (int rc = need_decodable(g)) return rc;
    fbgnn_ctx *ctx = g->ctx;
    if (set_device(ctx)) return FBGNN_E_CUDA;
    if (B == 0) return 0;
    SyndromeArgs a{g->dev, v2<const uint8_t>(noise), v2<uint8_t>(syndrome)};
    k_syndrome<<<(unsigned)B, 128, (size_t)g->dev.n, ctx->stream>>>(a);
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}

// ------------------------------------------------------------------ measurement helpers -
static int time_probe(fbgnn_ctx *ctx, void (*kernel)(float *, int), int iters, double per_thread_ops, double *rate) {
    float *d = nullptr;
    CK(cudaMalloc(&d, 4));
    const int blocks = ctx->num_sms * 8, threads = 256;
    kernel<<<blocks, threads, 0, ctx->stream>>>(d, 16);
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        CK(cudaEventRecord(ctx->ev0, ctx->stream));
        kernel<<<blocks, threads, 0, ctx->stream>>>(d, iters);
        CK(cudaEventRecord(ctx->ev1, ctx->stream));
        CK(cudaEventSynchronize(ctx->ev1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        best = std::min(best, ms);
        ctx->launches++;
    }
    CK(cudaGetLastError());
    CK(cudaFree(d));
    *rate = per_thread_ops * (double)blocks * threads / (best * 1e-3);
    return 0;
}

extern "C" int fbgnn_sfu_peak(fbgnn_ctx *ctx, double *evals_per_s) {
    REQUIRE(ctx && evals_per_s, "NULL argument");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    const int iters = 20000;
    return time_probe(ctx, k_sfu_peak, iters, 8.0 * iters, evals_per_s);
}

extern "C" int fbgnn_fma_peak(fbgnn_ctx *ctx, double *instr_per_s) {
    REQUIRE(ctx && instr_per_s, "NULL argument");
    if (set_device(ctx)) return FBGNN_E_CUDA;
    const int iters = 100000;
    return time_probe(ctx, k_fma_peak, iters, 8.0 * iters, instr_per_s);
}

extern "C" int fbgnn_math_probe(fbgnn_ctx *ctx, const char *fn, const float *x, float *y, int64_t n) {
    REQUIRE(ctx && fn && x && y && n >= 0, "bad argument");
    static const char *names[] = {"exp", "log", "log1p", "softplus", "phi4", "phi2", "tanh", "atanh", "mufu_ex2",
                                  "mufu_lg2", "sfu_exp", "sfu_log", "sfu_softplus", "sfu_phi4", "sfu_phi2", "mufu_rcp",
                                  "sfu_tanh", "sfu_atanh", nullptr, nullptr,
                                  // 20..24: scalar SFU building blocks; 25..31: their paired (float2) forms
                                  "sfu_exp2s", "sfu_logaddexp_open", "sfu_vn_corr", "sfu_vn_msg", "sfu_phi_open",
                                  "sfu2_exp2s", "sfu2_logaddexp_open", "sfu2_vn_corr", "sfu2_vn_msg", "sfu2_phi_open",
                                  "sfu2_softplus", "sfu2_tanh"};
    int id = -1;
    for (int i = 0; i < (int)(sizeof(names) / sizeof(names[0])); i++) if (names[i] && !std::strcmp(fn, names[i])) id = i;
    REQUIRE(id >= 0, "unknown probe function '%s'", fn);
    if (set_device(ctx)) return FBGNN_E_CUDA;
    if (n == 0) return 0;
    k_math_probe<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(id, x, y, n);
    CK(cudaGetLastError());
    ctx->launches++;
    return 0;
}
