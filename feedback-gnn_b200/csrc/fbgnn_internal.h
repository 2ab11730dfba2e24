// fbgnn_internal.h -- shared between the translation units of libfbgnn.so: error helpers, the
// handle structs behind the opaque types of include/fbgnn.h, and the launchers one unit offers another.
#pragma once
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/fbgnn.h"
#include "fbgnn_kernels.cuh"

using namespace fbgnn;

// ------------------------------------------------------------------ errors -------------
int fbgnn_fail(int code, const char *fmt, ...);      // sets the thread-local message, returns code (fbgnn_core.cu)
#define fail fbgnn_fail

#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess)                                                            \
            return fail(FBGNN_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                              \
    } while (0)

#define REQUIRE(cond, ...)                                   \
    do {                                                     \
        if (!(cond)) return fail(FBGNN_E_INVALID, __VA_ARGS__); \
    } while (0)


// ------------------------------------------------------------------ handles ------------
struct Workspace {                 // per-context scratch of the fused pipelines
    int64_t cap_frames = 0;
    int n = 0, m = 0;
    uint8_t *vbits = nullptr, *sbits = nullptr, *active[2] = {nullptr, nullptr}, *rounds = nullptr, *iters = nullptr;
    float *L = nullptr, *P = nullptr, *logit = nullptr;
    int *list[2] = {nullptr, nullptr};
    int *list_count = nullptr;     // [2]
    unsigned long long *counters = nullptr;   // [4]
    void *hard = nullptr;          // binary pipeline: unused (decisions live in vbits)
};

struct fbgnn_ctx {
    int device = 0, num_sms = 0;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int64_t launches = 0;
    int math_mode = FBGNN_MATH_EXACT;
    void *flush_buf = nullptr;
    size_t flush_bytes = 0;
    char name[256] = {0};
    Workspace ws;
    // communicator of the counter all-reduce (fbgnn_comm.cu); void* keeps nccl.h out of the other units
    void *comm = nullptr;
    int comm_rank = 0, comm_size = 1;
    void *comm_buf = nullptr;      // device staging buffer, FBGNN_COMM_MAX_ELEMS 8-byte elements
    int64_t collectives = 0;
    unsigned long long *stats = nullptr;   // device [2]: {frames, BP iterations executed} of the k_bp4 launches (fbgnn_ctx_stats)
};

struct fbgnn_graph {
    fbgnn_ctx *ctx;
    SideDev dev;
    int max_dc = 0, max_dv = 0;
    bool decodable = true;         // false: only the bit-packed rows exist (dense logical matrices)
    std::string why_not;
    std::vector<void *> allocs;
    std::vector<int> h_vn_ptr;     // host copy of the per-variable edge ranges
};

struct fbgnn_code {
    fbgnn_ctx *ctx;
    fbgnn_graph *X, *Z;
    int kx = 0, kz = 0, W = 0;
    uint32_t *lx_bits = nullptr, *lz_bits = nullptr;
    // host copies of the CSR of hx / hz (to cut row bases out of them) and the OSD-0 bases
    std::vector<int32_t> hx_ptr, hx_idx, hz_ptr, hz_idx;
    int *lx_ptr = nullptr, *lz_ptr = nullptr;                // CSR rows of the logical operators (GNN_BP4 logits)
    idx_t *lx_col = nullptr, *lz_col = nullptr;
    fbgnn_graph *basis_x = nullptr, *basis_z = nullptr;      // hx[pivot_hx], hz[pivot_hz]
    idx_t *pivot_x = nullptr, *pivot_z = nullptr;            // device [rank]
};

struct fbgnn_rows {
    fbgnn_ctx *ctx;
    int n = 0, m = 0;
    int *ptr = nullptr;            // device [m+1]
    idx_t *col = nullptr;          // device [nnz]
};

struct fbgnn_gnn {
    fbgnn_ctx *ctx;
    int H, M, act, reduce, use_bias;
    float *weights = nullptr;      // packed GnnLayout<H,M> (layers == 2) or the layer sequence of k_gnn_deep
    int total = 0;
    int layers = 2;                // num_mlp_layers
    float *w_tc = nullptr;         // tensor-core operand tiles + scalar block (tc::GnnW), H = 40 / M = 20 only
    int gemm = FBGNN_GEMM_FMA;     // FBGNN_GEMM_*: how the dense products of the node update are evaluated
};


static inline int set_device(fbgnn_ctx *ctx) {
    CK(cudaSetDevice(ctx->device));
    return 0;
}

static inline int need_decodable(const fbgnn_graph *g) {
    if (!g->decodable) return fail(FBGNN_E_UNSUPPORTED, "%s", g->why_not.c_str());
    return 0;
}

template <typename T> static View2<T> v2(const fbgnn_tensor2 &t) { return View2<T>{(T *)t.ptr, t.s0, t.s1}; }
template <typename T> static View3<T> v3(const fbgnn_tensor3 &t) { return View3<T>{(T *)t.ptr, t.s0, t.s1, t.s2}; }


template <typename K>
static int set_smem(K kernel, size_t bytes, fbgnn_ctx *ctx, const char *what) {
    if (bytes > ctx->smem_optin)
        return fail(FBGNN_E_UNSUPPORTED, "%s needs %zu bytes of shared memory per frame, the device offers %zu",
                    what, bytes, ctx->smem_optin);
    if (bytes > 48 * 1024) CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return 0;
}

void ws_free(Workspace &w);                                              // fbgnn_core.cu
// launchers shared between units
int launch_bp4(fbgnn_ctx *ctx, const Bp4Args &a, int64_t grid);          // fbgnn_bp.cu
int launch_bp2(fbgnn_ctx *ctx, const Bp2Args &a, int64_t B);             // fbgnn_bp.cu
int launch_gnn(fbgnn_ctx *ctx, const fbgnn_gnn *g, GnnArgs &a);          // fbgnn_gnn.cu
int launch_osd(fbgnn_ctx *ctx, OsdArgs &a, int order, int64_t grid);    // fbgnn_pipeline.cu
