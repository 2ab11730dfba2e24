/* fbgnn.h -- C ABI of libfbgnn.so: the B200 (sm_100a) implementation of Feedback-GNN's
 * BP -> feedback-GNN -> BP hot path.
 *
 * The reference (gongaa/Feedback-GNN) has no FFI of its own: its "operator API" for this
 * path is the Python call surface of a handful of Keras layers/models.  Each entry point
 * below is what a binding for one of those calls needs; the Python host side
 * (feedback-gnn_b200/fbgnn/) binds them with ctypes and mirrors the reference classes.
 *
 *   fbgnn_code_create        <- css_code / QLDPCBPDecoder.__init__ edge tables
 *                               sionna/fec/ldpc/codes_q.py:8-49, decoding_q.py:58-94
 *   fbgnn_graph_create       <- LDPCBPDecoder.__init__ edge tables       decoding.py:325-347
 *   fbgnn_bp4_decode         <- QLDPCBPDecoder.call                      decoding_q.py:661-797
 *   fbgnn_bp2_decode         <- LDPCBPDecoder.call (is_syndrome)         decoding.py:875-1048
 *   fbgnn_gnn_create/_forward<- Feedback_GNN.build / .call, set_weights  feedback_gnn.py:110-188
 *   fbgnn_pauli_sample       <- Pauli.call (non-wt branch)               channel/pauli.py:98-108
 *   fbgnn_bsc_sample         <- BinarySymmetricChannel.call              channel/discrete_channel.py:385-396
 *   fbgnn_syndrome           <- int_mod_2(tf.matmul(H, noise))           feedback_gnn.py:308-309
 *   fbgnn_osd0_decode        <- OSD0_Decoder.call                        bp_osd.py:8-77
 *   fbgnn_osd_decode         <- OSD0_Decoder.call + the OSD-CS sweep (Roffe et al. 2020; ldpc's osd_cs)
 *   fbgnn_gbp_create/_decode <- GNN_BP4.build / .call                    gnn.py:71-420
 *   fbgnn_pipeline_run       <- Sandwich_BP_GNN_Evaluation_Model.call    feedback_gnn.py:293-361
 *   fbgnn_bsc_pipeline_run   <- BP_BSC_Model.call                        feedback_gnn.py:207-229
 *
 * Conventions
 *   - Every function returns 0 on success or a negative FBGNN_E_* code; the message is
 *     available from fbgnn_last_error() (thread-local).  No exception crosses the ABI.
 *   - Handles are opaque, created/destroyed by the caller, and not thread-safe
 *     individually: use one context per GPU per host thread.
 *   - All tensor arguments are DEVICE pointers on the context's GPU (the host side moves
 *     numpy arrays with fbgnn_memcpy_* and exchanges device tensors zero-copy via DLPack);
 *     they are borrowed for the duration of the call.  A tensor is described by its base
 *     pointer and explicit ELEMENT strides (fbgnn_tensor2/3), so the reference's layouts
 *     ([B,3,n] priors, [m,B] syndromes/logits, transposed views) need no copies.
 *   - Work is enqueued on the context's stream; functions that return host data
 *     synchronise that stream, the others are asynchronous (fbgnn_ctx_sync to wait).
 *   - There is no CPU fallback: without a CUDA device every compute entry point fails
 *     with FBGNN_E_CUDA.
 */
#ifndef FBGNN_H
#define FBGNN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FBGNN_VERSION 200            /* 0.2.0 */

#define FBGNN_OK            0
#define FBGNN_E_INVALID    -1        /* bad argument */
#define FBGNN_E_CUDA       -2        /* CUDA runtime error (message has the detail) */
#define FBGNN_E_UNSUPPORTED -3       /* valid request this build cannot serve (e.g. code too large) */
#define FBGNN_E_NOMEM      -4

/* check-node update of the BP decoders (cn_type of the reference's decoders) */
#define FBGNN_CN_PHI     0           /* "boxplus-phi" */
#define FBGNN_CN_TANH    1           /* "boxplus"     */
#define FBGNN_CN_MINSUM  2           /* "minsum"      */

/* arithmetic of the decoders (fbgnn_ctx_set_math) */
#define FBGNN_MATH_EXACT 0           /* exp / log as polynomials on the FP32 pipe (1 ulp)                              */
#define FBGNN_MATH_SFU   1           /* exp / log on the special-function unit (MUFU.EX2 / LG2, 2-3 ulp), ~2.3x fewer   */
                                     /* instructions; both are bit-identical to the CPU oracle in the same arithmetic  */
#define FBGNN_MATH_FAST  FBGNN_MATH_SFU   /* former name */

/* Feedback_GNN options */
#define FBGNN_ACT_TANH   0
#define FBGNN_ACT_RELU   1
#define FBGNN_ACT_LINEAR 2
#define FBGNN_GEMM_FMA    0           /* GNN_BP4 matrix products in FP32 FMAs, bit-exact with the oracle (default) */
#define FBGNN_GEMM_TF32X3 1           /* on tcgen05 tensor cores, 3-product TF32 split: float32 accuracy; other bits than the FMA form */
#define FBGNN_REDUCE_MEAN 0
#define FBGNN_REDUCE_SUM  1
#define FBGNN_REDUCE_MAX  2
#define FBGNN_REDUCE_MIN  3

typedef struct fbgnn_ctx   fbgnn_ctx;     /* one GPU: stream, scratch, timers            */
typedef struct fbgnn_graph fbgnn_graph;   /* Tanner graph of one parity-check matrix     */
typedef struct fbgnn_code  fbgnn_code;    /* CSS code: graphs of hx, hz + logicals lx,lz */
typedef struct fbgnn_gnn   fbgnn_gnn;     /* one Feedback_GNN weight set                 */
typedef struct fbgnn_gbp   fbgnn_gbp;     /* one GNN_BP4 weight set                      */
typedef struct fbgnn_rows  fbgnn_rows;    /* sparse rows of a binary matrix (soft-syndrome row sets) */

/* strided views (strides in ELEMENTS; ptr == NULL means "absent") */
typedef struct { void *ptr; int64_t s0, s1; } fbgnn_tensor2;
typedef struct { void *ptr; int64_t s0, s1, s2; } fbgnn_tensor3;

/* ---- library / context ------------------------------------------------------------ */
int fbgnn_version(void);
const char *fbgnn_last_error(void);
int fbgnn_device_count(int *count);
int fbgnn_ctx_create(int device, fbgnn_ctx **ctx);
int fbgnn_ctx_destroy(fbgnn_ctx *ctx);
int fbgnn_ctx_sync(fbgnn_ctx *ctx);
int fbgnn_ctx_device(fbgnn_ctx *ctx, int *device, int *num_sms, char *name, int name_len);
/* CUDA-event timer on the context's stream (what bench.py times kernels with) */
int fbgnn_timer_start(fbgnn_ctx *ctx);
int fbgnn_timer_stop(fbgnn_ctx *ctx, float *elapsed_ms);          /* synchronises */
/* Arithmetic mode used by the kernels this context launches from now on (FBGNN_MATH_*). */
int fbgnn_ctx_set_math(fbgnn_ctx *ctx, int32_t mode);
int fbgnn_ctx_get_math(fbgnn_ctx *ctx, int32_t *mode);
/* Executed-work counters of the quaternary BP launches of this context: out = {frames decoded, BP iterations actually
 * executed} since the last reset (the fixed-point exit skips iterations; bench.py reports its roofline on the work
 * executed).  The first call switches the counting on (two atomics per frame); out may be NULL. */
int fbgnn_ctx_stats(fbgnn_ctx *ctx, int64_t out[2], int32_t reset);
/* number of kernel launches this context has enqueued so far */
int fbgnn_launch_count(fbgnn_ctx *ctx, int64_t *launches);

/* ---- memory ------------------------------------------------------------------------ */
int fbgnn_malloc(fbgnn_ctx *ctx, size_t bytes, void **dptr);
int fbgnn_free(fbgnn_ctx *ctx, void *dptr);
int fbgnn_memset(fbgnn_ctx *ctx, void *dptr, int value, size_t bytes);             /* async */
int fbgnn_memcpy_h2d(fbgnn_ctx *ctx, void *dst, const void *src, size_t bytes);   /* async w.r.t. host only for pinned src */
int fbgnn_memcpy_d2h(fbgnn_ctx *ctx, void *dst, const void *src, size_t bytes);   /* synchronises */
int fbgnn_memcpy_d2d(fbgnn_ctx *ctx, void *dst, const void *src, size_t bytes);   /* async */
int fbgnn_host_alloc(size_t bytes, void **hptr);                                  /* pinned */
int fbgnn_host_free(void *hptr);
/* write a buffer larger than L2 (bench.py uses it between timed iterations) */
int fbgnn_flush_l2(fbgnn_ctx *ctx);

/* ---- code / graph ------------------------------------------------------------------- */
/* CSR of a binary matrix: indptr[rows+1], indices[nnz] (column indices, increasing per row),
 * host pointers, copied. */
int fbgnn_graph_create(fbgnn_ctx *ctx, int32_t n, int32_t m, const int32_t *indptr,
                       const int32_t *indices, fbgnn_graph **graph);
int fbgnn_graph_destroy(fbgnn_graph *graph);
/* hx [m_x,n], hz [m_z,n], logical operators lx [k_x,n], lz [k_z,n], all CSR, host pointers */
int fbgnn_code_create(fbgnn_ctx *ctx, int32_t n,
                      int32_t m_x, const int32_t *hx_indptr, const int32_t *hx_indices,
                      int32_t m_z, const int32_t *hz_indptr, const int32_t *hz_indices,
                      int32_t k_x, const int32_t *lx_indptr, const int32_t *lx_indices,
                      int32_t k_z, const int32_t *lz_indptr, const int32_t *lz_indices,
                      fbgnn_code **code);
int fbgnn_code_destroy(fbgnn_code *code);
/* Row bases for OSD-0: pivot_hx[rank_x] / pivot_hz[rank_z] are the rows of hx / hz that form a basis
 * (css_code.pivot_hx / pivot_hz, codes_q.py:36-39).  Needed before a pipeline with cfg.osd0. */
int fbgnn_code_set_basis(fbgnn_code *code, int32_t rank_x, const int32_t *pivot_hx, int32_t rank_z,
                         const int32_t *pivot_hz);
/* number of edges of hx and hz (message array lengths) */
int fbgnn_code_edges(fbgnn_code *code, int32_t *e_x, int32_t *e_z);

/* ---- noise sources ------------------------------------------------------------------- */
/* Pauli.call, non-wt branch.  thr = {px, px - py, (px + pz) - py} as float32.  Uniforms
 * come from Philox4x32-10: key = seed, counter = (global frame id, qubit/4, stream 0).
 * noise_x/noise_z: uint8 [B,n] views. */
int fbgnn_pauli_sample(fbgnn_ctx *ctx, int32_t n, int64_t B, const float thr[3], uint64_t seed,
                       uint64_t first_frame, fbgnn_tensor2 noise_x, fbgnn_tensor2 noise_z);
/* Pauli.call, wt branch (pauli.py:80-96): exactly `wt` erroneous qubits per frame (partial
 * Fisher-Yates from Philox stream 2), each X, Y or Z with probability 1/3 (stream 3). */
int fbgnn_pauli_sample_wt(fbgnn_ctx *ctx, int32_t n, int64_t B, int32_t wt, uint64_t seed,
                          uint64_t first_frame, fbgnn_tensor2 noise_x, fbgnn_tensor2 noise_z);
/* Bernoulli(p) flips (stream 1 of the same generator). noise: uint8 [B,n] */
int fbgnn_bsc_sample(fbgnn_ctx *ctx, int32_t n, int64_t B, float p, uint64_t seed,
                     uint64_t first_frame, fbgnn_tensor2 noise);
/* syndrome[c,b] = XOR_{v in row c} noise[b,v].  noise: uint8 view indexed (b,v);
 * syndrome: uint8 view indexed (c,b). */
int fbgnn_syndrome(fbgnn_graph *graph, int64_t B, fbgnn_tensor2 noise, fbgnn_tensor2 syndrome);

/* ---- decoders ------------------------------------------------------------------------ */
/* QLDPCBPDecoder.call.
 *   llr        float32 view indexed (b, k in {x,y,z}, v); NULL ptr -> constant `prior`
 *   synd_x/z   uint8 views indexed (c, b)
 *   Lx,Ly,Lz   float32 views indexed (b, v)                       (marginals)
 *   x_hat,z_hat uint8 views indexed (b, v)                        (argmin decision)
 *   x_logit    float32 view indexed (row of hz, b), z_logit (row of hx, b): the stage_one
 *              soft syndromes; NULL ptr -> not computed
 *   msg_x/msg_z float32 views indexed (b, edge) receiving the final check-to-variable
 *              messages in VN-sorted edge order (teacher-forced parity tests); NULL -> skipped
 *   iter_logits float32 view indexed (slot, row, b), 2*num_iter+2 slots: the soft syndromes before
 *              every iteration and after the last -- the llr_hat of the reference's stage_two /
 *              trainable mode (decoding_q.py:730, 743-746, 779-781); NULL -> skipped
 */
int fbgnn_bp4_decode(fbgnn_code *code, int32_t cn_type, int32_t num_iter, float factor, int64_t B,
                     fbgnn_tensor3 llr, float prior, fbgnn_tensor2 synd_x, fbgnn_tensor2 synd_z,
                     fbgnn_tensor2 Lx, fbgnn_tensor2 Ly, fbgnn_tensor2 Lz,
                     fbgnn_tensor2 x_hat, fbgnn_tensor2 z_hat,
                     fbgnn_tensor2 x_logit, fbgnn_tensor2 z_logit,
                     fbgnn_tensor2 msg_x, fbgnn_tensor2 msg_z, fbgnn_tensor3 iter_logits);

/* Rows of a binary matrix as CSR on the device (any density; at most 65535 columns): the row sets over which
 * fbgnn_bp4_decode_ex forms soft syndromes. */
int fbgnn_rows_create(fbgnn_ctx *ctx, int32_t n, int32_t m, const int32_t *indptr, const int32_t *indices,
                      fbgnn_rows **rows);
int fbgnn_rows_destroy(fbgnn_rows *rows);

/* Options of fbgnn_bp4_decode_ex (zero-initialise; every field optional). */
typedef struct {
    /* OPT-IN early stop (SURVEY.md H8).  The reference always runs num_iter iterations (decoding_q.py:732).  With
     * iters_out != NULL a frame leaves the loop as soon as the hard decision of its current messages reproduces the
     * syndrome (checked after every iteration by a warp ballot over the checks); iters_out[b] (device uint8 [B],
     * num_iter <= 255) receives the iterations executed, and the frame's outputs are exactly those of a decoder
     * configured with num_iter = iters_out[b]. */
    uint8_t *iters_out;
    /* Row sets of the soft syndromes: x_logit over rows_x (from llr_x'), z_logit over rows_z (from llr_z').  NULL =
     * the rows of hz / hx (the stage_one / stage_two choice, decoding_q.py:35-37); the reference's trainable mode
     * without those flags uses the dense hx_perp / hz_perp (decoding_q.py:32-33, 93-94). */
    fbgnn_rows *rows_x, *rows_z;
} fbgnn_bp4_opts;

/* fbgnn_bp4_decode with options; x_logit / z_logit / iter_logits are then indexed by the rows of opts->rows_x / rows_z. */
int fbgnn_bp4_decode_ex(fbgnn_code *code, int32_t cn_type, int32_t num_iter, float factor, int64_t B,
                        fbgnn_tensor3 llr, float prior, fbgnn_tensor2 synd_x, fbgnn_tensor2 synd_z,
                        fbgnn_tensor2 Lx, fbgnn_tensor2 Ly, fbgnn_tensor2 Lz,
                        fbgnn_tensor2 x_hat, fbgnn_tensor2 z_hat,
                        fbgnn_tensor2 x_logit, fbgnn_tensor2 z_logit,
                        fbgnn_tensor2 msg_x, fbgnn_tensor2 msg_z, fbgnn_tensor3 iter_logits,
                        const fbgnn_bp4_opts *opts);

/* LDPCBPDecoder.call with is_syndrome.  llr: float32 logits (b,v); synd: uint8 (c,b) or
 * NULL ptr (no syndrome); soft: float32 (b,v) output logits; hard: uint8 (b,v) or NULL. */
int fbgnn_bp2_decode(fbgnn_graph *graph, int32_t cn_type, int32_t num_iter, float factor,
                     int64_t B, fbgnn_tensor2 llr, fbgnn_tensor2 synd, fbgnn_tensor2 soft,
                     fbgnn_tensor2 hard);

/* The same with the reference's optional decoder features: edge_weights (device float32 [E], edges sorted by
 * (variable, check); NULL = none) multiply the variable-to-check messages (trainable=True, decoding.py:361-366,
 * 981-983); msg_in / msg_out (float32 views (b, edge), NULL ptr = absent) carry the check-to-variable messages into
 * and out of the call (stateful=True, decoding.py:947-953, 1045-1048). */
int fbgnn_bp2_decode_ex(fbgnn_graph *graph, int32_t cn_type, int32_t num_iter, float factor, int64_t B,
                        fbgnn_tensor2 llr, fbgnn_tensor2 synd, fbgnn_tensor2 soft, fbgnn_tensor2 hard,
                        const float *edge_weights, fbgnn_tensor2 msg_in, fbgnn_tensor2 msg_out);

/* OSD0_Decoder.call (bp_osd.py:51-77): ordered-statistics post-processing of order 0.  `basis` is the
 * graph of a FULL-RANK row basis of the parity-check matrix (rank rows); llr float32 (b, v) are the
 * reliabilities BP produced (small = likely in error; ties are broken by index); synd uint8 (row, b) is
 * the syndrome reduced to the basis rows; e_hat uint8 (b, v) receives the error that satisfies it. */
int fbgnn_osd0_decode(fbgnn_graph *basis, int64_t B, fbgnn_tensor2 llr, fbgnn_tensor2 synd,
                      fbgnn_tensor2 e_hat);
/* Ordered-statistics decoding of order `order` with the combination sweep (OSD-CS; Roffe et al., "Decoding
 * across the quantum LDPC code landscape", 2020; the `ldpc` package's osd_method="osd_cs").  Arguments as
 * fbgnn_osd0_decode; order 0 is OSD-0, bit for bit.  With order lam > 0 the elimination of OSD-0 is followed,
 * on the same reduced matrix, by a sweep over candidate sets T of the non-pivot columns c_0 < c_1 < ...
 * (least reliable first): index 0 the empty set, 1 + i the single {c_i}, then the pairs {c_i, c_j},
 * i < j < min(lam, n - rank), in lexicographic order.  T's solution is 1 on T and on pivot r the reduced
 * syndrome bit XOR the columns of T in row r; the candidate of least (Hamming weight, index) is returned, so
 * the result is the OSD-0 solution unless a candidate is strictly lighter.  order outside [0, 65535]:
 * FBGNN_E_INVALID.  A frame's reduced matrix lives in the shared memory of one CTA or, when it does not fit there,
 * is split by rows over a thread-block cluster of 2, 4 or 8 CTAs (same result, bit for bit); a basis that does
 * not fit a cluster of 8 either returns FBGNN_E_UNSUPPORTED, with the bytes it needs in the message. */
int fbgnn_osd_decode(fbgnn_graph *basis, int32_t order, int64_t B, fbgnn_tensor2 llr, fbgnn_tensor2 synd,
                     fbgnn_tensor2 e_hat);

/* Localised statistics decoding of order 0 (LSD-0; Hillmann, Berent, Quintavalle, Eisert, Wille, Roffe, 2024; the
 * `ldpc` package's BpLsdDecoder) on any parity-check matrix `pcm` (R rows; the full hx / hz or an OSD basis).  Clusters
 * grow around the unsatisfied checks, one column per invalid cluster and round, taking the least reliable column
 * (ascending llr, ties by index, -0.0 before +0.0) next to the cluster; clusters that meet are united; a cluster stops
 * growing once its syndrome lies in the span of its columns, and each is then solved as OSD-0 would solve it
 * (csrc/fbgnn_lsd.cuh and DESIGN.md §4 give the exact definition).  llr float32 (b, v), synd uint8 (row, b) over all R
 * rows, e_hat uint8 (b, v) (optional: NULL ptr skips it).  max_cols / max_checks bound the columns and checks of all clusters of a frame together
 * (0 = defaults 256 / 256; limits 512 / 512, outside [1, limit]: FBGNN_E_INVALID).  status (optional, device uint8
 * [B]): 0 solved (pcm e_hat = synd), 1 abandoned over budget, 2 abandoned because the syndrome is outside the column
 * space of pcm; an abandoned frame gets e_hat = 0.  One CTA per frame; works for every graph fbgnn_graph_create
 * accepts. */
int fbgnn_lsd_decode(fbgnn_graph *pcm, int32_t max_cols, int32_t max_checks, int64_t B, fbgnn_tensor2 llr,
                     fbgnn_tensor2 synd, fbgnn_tensor2 e_hat, uint8_t *status);

/* ---- feedback GNN --------------------------------------------------------------------- */
/* Weights in Keras get_weights() order, host float32 pointers (copied); bias pointers may
 * be NULL when use_bias is False.  Shapes: W0[H,3] b0[3] W1x[4,H] b1x[H] W2x[H,M] b2x[M]
 * W1z[4,H] b1z[H] W2z[H,M] b2z[M] W3[2M+3,H] b3[H]: the 2-layer MLPs of the shipped weights (tuned kernel). */
int fbgnn_gnn_create(fbgnn_ctx *ctx, int32_t H, int32_t M, int32_t activation, int32_t reduce_op,
                     const float *W0, const float *b0, const float *W1x, const float *b1x,
                     const float *W2x, const float *b2x, const float *W1z, const float *b1z,
                     const float *W2z, const float *b2z, const float *W3, const float *b3,
                     fbgnn_gnn **gnn);
/* Feedback_GNN with num_mlp_layers != 2 (feedback_gnn.py:110-127), any hidden / message dims up to 128.  `packed`:
 * the dense layers one after the other, each [K_in x K_out] row-major followed by K_out biases (zeros without bias):
 * _llr_inv_embed ((L == 1 ? 2M+3 : H) -> 3), vn_msg_mlp_x (4 -> H ... -> M, L layers), vn_msg_mlp_z, vn_embed_mlp
 * (2M+3 -> H ... -> H, L-1 layers) -- the Keras get_weights() order.  Runs through fbgnn_gnn_forward / the pipelines. */
int fbgnn_gnn_create_deep(fbgnn_ctx *ctx, int32_t H, int32_t M, int32_t num_mlp_layers, int32_t activation,
                          int32_t reduce_op, int32_t use_bias, const float *packed, int64_t count, fbgnn_gnn **gnn);
int fbgnn_gnn_destroy(fbgnn_gnn *gnn);
/* Select how the dense products of the node update (hidden sums x W2x / W2z, messages x W3) are evaluated (FBGNN_GEMM_*).
 * FBGNN_GEMM_TF32X3 runs them on the tcgen05 tensor cores with the three-product TF32 split (csrc/fbgnn_gnn_tc.cuh):
 * float32 re-association accuracy (5e-7 from the default FMA form); the oracle reproduces it bit for bit through the integer
 * model of a tcgen05.mma step (csrc/fb_umma.h).  Built for H = 40, M = 20,
 * 2-layer MLPs, tanh, reduce_op mean / sum and (3, .)-regular codes; otherwise FBGNN_E_UNSUPPORTED. */
int fbgnn_gnn_set_gemm(fbgnn_gnn *gnn, int32_t mode);
/* Feedback_GNN.call.  h_vn float32 (b, v, k); logit_hx (row of hx, b), logit_hz (row of hz, b);
 * synd_x/z uint8 (c, b); out float32 (b, v, k). */
int fbgnn_gnn_forward(fbgnn_code *code, fbgnn_gnn *gnn, int64_t B, fbgnn_tensor3 h_vn,
                      fbgnn_tensor2 logit_hx, fbgnn_tensor2 logit_hz, fbgnn_tensor2 synd_x,
                      fbgnn_tensor2 synd_z, fbgnn_tensor3 out);

/* ---- GNN_BP4: the full GNN message-passing decoder (gnn.py:71-751, BASELINE configs[4]) -------- */
/* arrays: 30 host float32 pointers in Keras get_weights() order (biases NULL when use_bias is False):
 *   [0,1]   _llr_inv_embed            kernel [d,3], bias [3]
 *   [2..9]  update_h_cn._msg_mlp_x/_z  (W1 [2d,H], b1 [H], W2 [H,M], b2 [M]) x 2
 *   [10..17] update_h_cn._embed_mlp_x/_z (W1 [M+d+1,H], b1, W2 [H,d], b2 [d]) x 2
 *   [18..25] update_h_vn._msg_mlp_x/_z  (as above)
 *   [26..29] update_h_vn._embed_mlp     (W1 [2M+d,H], b1, W2 [H,d], b2 [d])
 * This build provides num_embed_dims/num_hidden_units/num_msg_dims = 20/40/20, 2-layer MLPs, no attributes. */
int fbgnn_gbp_create(fbgnn_ctx *ctx, int32_t d, int32_t H, int32_t M, int32_t activation, int32_t reduce_op,
                     const float *const *arrays, fbgnn_gbp **gbp);
int fbgnn_gbp_destroy(fbgnn_gbp *gbp);
/* ---- training: second stage (widening into SURVEY.md section 8(f) N3) ------------------ */
/* Loss and weight gradients of Second_Stage_GNN_BP_Model.call under tf.GradientTape
 * (feedback_gnn.py:395-460; training loop examples/Feedback_GNN.ipynb cells 2 and 8):
 *   new priors = Feedback_GNN(h_vn, logit_hx, logit_hz, synd_x, synd_z);  BP4 (boxplus-phi, `num_iter`
 *   iterations, `factor`) with the soft syndromes of every iteration;
 *   loss = sum_{i=loss_from}^{num_iter-1} bce(1 - synd_z, x_logit_{i+1}) + bce(1 - synd_x, z_logit_{i+1}).
 * Inputs as fbgnn_gnn_forward.  *loss (host) receives the loss; with want_grad != 0, grads (host, 3923
 * floats) receives d loss / d weights as the row-major blocks [W0; b0] (41x3), [W1x; b1x] (5x40),
 * [W2x; b2x] (41x20), [W1z; b1z], [W2z; b2z], [W3; b3] (44x40).  Synchronises the stream. */
int fbgnn_second_stage_grad(fbgnn_code *code, fbgnn_gnn *gnn, int32_t num_iter, float factor, int32_t loss_from,
                            int64_t B, fbgnn_tensor3 h_vn, fbgnn_tensor2 logit_hx, fbgnn_tensor2 logit_hz,
                            fbgnn_tensor2 synd_x, fbgnn_tensor2 synd_z, int32_t want_grad, double *loss,
                            float *grads);

/* Select how GNN_BP4's per-node matrix products are evaluated (FBGNN_GEMM_*).  The tensor-core form
 * (fbgnn_gbp_tc.cuh) needs reduce_op mean / sum and tanh; otherwise FBGNN_E_UNSUPPORTED. */
int fbgnn_gbp_set_gemm(fbgnn_gbp *gbp, int32_t mode);
/* The embeddings of a batch live in HBM ((n + m)(d + H) + n H floats per frame); fbgnn_gbp_decode walks the batch
 * in chunks of a few GB.  max_frames > 0 caps the chunk (tests force several chunks with a ragged tail); 0 = automatic. */
int fbgnn_gbp_set_chunk(fbgnn_gbp *gbp, int64_t max_frames);
/* GNN_BP4.call: synd_x uint8 [B,m_x], synd_z uint8 [B,m_z] contiguous, batch first (gnn.py:385-386);
 * x_logit float32 (iteration, row, b) with m_z + k_z rows = [hz_logit; lz_logit], z_logit with m_x + k_x rows
 * = [hx_logit; lx_logit] (either may be NULL); x_hat, z_hat uint8 (v, b): the argmin decision. */
int fbgnn_gbp_decode(fbgnn_code *code, fbgnn_gbp *gbp, int32_t num_iter, int64_t B, fbgnn_tensor2 synd_x,
                     fbgnn_tensor2 synd_z, fbgnn_tensor3 x_logit, fbgnn_tensor3 z_logit, fbgnn_tensor2 x_hat,
                     fbgnn_tensor2 z_hat);

/* ---- fused Monte-Carlo pipelines ------------------------------------------------------- */
typedef struct {
    int32_t num_stages;        /* num_layers of the reference = 1 + GNN rounds              */
    const int32_t *num_iter;   /* [num_stages] host                                          */
    const float *factor;       /* [num_stages] host                                          */
    const int32_t *cn_type;    /* [num_stages] host                                          */
    fbgnn_gnn *const *gnn;     /* [num_stages-1] host array of handles                       */
    float prior;               /* log(3(1-p0)/p0) as float32                                 */
    float thr[3];              /* Pauli thresholds, see fbgnn_pauli_sample                   */
    int32_t fixed_weight;      /* > 0: errors of exactly this weight (Pauli wt=True) instead  */
    int32_t osd0;              /* 1: OSD-0 on the frames still mismatching after the last stage */
                               /*    (BP4_OSD_Model, bp_osd.py:80-197)                          */
    int32_t skip_inactive;     /* 0: all frames run all rounds (reference-equivalent work)   */
                               /* 1: frames whose decision matches the syndrome stop early   */
                               /*    (result-identical; the reference masks the scatter)     */
    int32_t early_stop;        /* 1: OPT-IN early stop inside every BP stage (see fbgnn_bp4_opts; NOT result-identical */
                               /*    to the reference in general -- a converged frame keeps its first converged state)  */
    int32_t osd_order;         /* with osd0: 0 = OSD-0, lam in [1, 65535] = OSD-CS of order lam (fbgnn_osd_decode),     */
                               /*    the same order on both sides (basis_x with osd_llrz, basis_z with osd_llrx)       */
    int32_t lsd;               /* with osd0: 1 = re-solve the frames still mismatching with LSD-0 (fbgnn_lsd_decode)   */
                               /*    instead of OSD, on each side's full matrix (hx with osd_llrz and the full         */
                               /*    syndrome_x, hz with osd_llrx); no fbgnn_code_set_basis needed; a side LSD-0       */
                               /*    abandons keeps its BP decision                                                     */
    int32_t lsd_max_cols, lsd_max_checks;   /* LSD-0 budgets (0 = defaults), as fbgnn_lsd_decode                       */
} fbgnn_pipeline_cfg;

/* Sandwich_BP_GNN_Evaluation_Model.call on global frames [first_frame, first_frame+B).
 *   noise_x/noise_z  optional uint8 (b,v) device views used instead of sampling
 *   flags            optional uint8 [B] device: bit0 flagged, bit1 block error,
 *                    bits 2..7 number of GNN rounds the frame was active in
 *   x_diff/z_diff    optional uint8 (b,v) device views: residual error after correction
 *   counters         optional HOST int64[4]: {frames, flagged, block errors, frames that
 *                    failed stage 0}; when given, the call synchronises
 */
int fbgnn_pipeline_run(fbgnn_code *code, const fbgnn_pipeline_cfg *cfg, uint64_t seed,
                       uint64_t first_frame, int64_t B, fbgnn_tensor2 noise_x,
                       fbgnn_tensor2 noise_z, uint8_t *flags, fbgnn_tensor2 x_diff,
                       fbgnn_tensor2 z_diff, int64_t *counters);

/* The same pipeline with PACKED inputs and outputs (32 qubits / 32 frames per word; what a Monte-Carlo host loop needs
 * is 8x smaller than byte arrays and the loads / stores are whole words):
 *   noise_x_bits / noise_z_bits  optional uint32 [B][wq] device, wq = (ceil(n / 32) rounded up to 4): qubit v of frame b is
 *                    bit (v & 31) of word [b][v >> 5]; NULL = sample in-kernel
 *   frame_bits       optional uint32 [3][ceil(B / 32)] device: planes {flagged, block error, failed stage 0}, frame b is
 *                    bit (b & 31) of word b >> 5
 *   x_diff_bits / z_diff_bits  optional uint32 [B][wq] device: residual error after correction, packed like the noise */
int fbgnn_pipeline_run_bits(fbgnn_code *code, const fbgnn_pipeline_cfg *cfg, uint64_t seed, uint64_t first_frame,
                            int64_t B, const uint32_t *noise_x_bits, const uint32_t *noise_z_bits,
                            uint32_t *frame_bits, uint32_t *x_diff_bits, uint32_t *z_diff_bits, int64_t *counters);

/* BP_BSC_Model.call: Bernoulli(p) noise, syndrome with `graph`, binary BP from the constant
 * logit llr_const, residual syndrome + logical check against `logical` (block error = any row of
 * `logical` . residual; NULL: block error = flagged).  flags/counters as above.
 * osd_basis / osd_pivot (optional): BP2_OSD_Model (bp_osd.py:199-274) -- the frames whose decision
 * misses the syndrome are re-solved by OSD-0 on the given row basis (osd_pivot: HOST int32 rows of
 * `graph` behind the basis rows). */
int fbgnn_bsc_pipeline_run(fbgnn_graph *graph, fbgnn_graph *logical, int32_t cn_type,
                           int32_t num_iter, float factor, float llr_const, float p, uint64_t seed,
                           uint64_t first_frame, int64_t B, fbgnn_tensor2 noise, uint8_t *flags,
                           int64_t *counters, fbgnn_graph *osd_basis, const int32_t *osd_pivot);
/* The same with OSD of order osd_order on the failed frames (0 = OSD-0, lam = OSD-CS; fbgnn_osd_decode). */
int fbgnn_bsc_pipeline_run_ex(fbgnn_graph *graph, fbgnn_graph *logical, int32_t cn_type,
                              int32_t num_iter, float factor, float llr_const, float p, uint64_t seed,
                              uint64_t first_frame, int64_t B, fbgnn_tensor2 noise, uint8_t *flags,
                              int64_t *counters, fbgnn_graph *osd_basis, const int32_t *osd_pivot,
                              int32_t osd_order);
/* The same with LSD-0 (fbgnn_lsd_decode, sign -1: the binary decoder's logits) on `graph` itself for the failed frames,
 * with the budgets max_cols / max_checks (0 = defaults); an abandoned frame keeps its BP decision. */
int fbgnn_bsc_pipeline_run_lsd(fbgnn_graph *graph, fbgnn_graph *logical, int32_t cn_type,
                               int32_t num_iter, float factor, float llr_const, float p, uint64_t seed,
                               uint64_t first_frame, int64_t B, fbgnn_tensor2 noise, uint8_t *flags,
                               int64_t *counters, int32_t max_cols, int32_t max_checks);

/* ---- multi-GPU: the one collective of the path (SURVEY.md 8(e)) ------------------------- */
/* Monte-Carlo frames shard across the GPUs of a box by global frame id; nothing but the counters is
 * ever exchanged.  One process per GPU: rank 0 makes an id (fbgnn_comm_unique_id), hands the 128 bytes
 * to the other ranks by any host channel (fbgnn/distributed.py uses a rendezvous file), and every rank
 * attaches its context with fbgnn_comm_init_rank (ncclCommInitRank; collective).  NCCL is bound at run
 * time (libnccl.so.2, or $FBGNN_NCCL_LIB); a context without a communicator is a 1-rank job and the
 * reductions below are identities.  The reference has no counterpart (one process per --gpu_id,
 * n1270.py:10-26); the host loop that needs the global counters is sim_ber's stopping rule
 * (sionna/utils/misc.py:710-716). */
#define FBGNN_COMM_ID_BYTES 128
#define FBGNN_COMM_MAX_ELEMS 64
#define FBGNN_RED_SUM 0
#define FBGNN_RED_MAX 1
int fbgnn_comm_unique_id(uint8_t id[FBGNN_COMM_ID_BYTES]);
int fbgnn_comm_init_rank(fbgnn_ctx *ctx, int32_t nranks, int32_t rank, const uint8_t id[FBGNN_COMM_ID_BYTES]);
int fbgnn_comm_info(fbgnn_ctx *ctx, int32_t *nranks, int32_t *rank, int32_t *nccl_version);
/* in-place sum over ranks of HOST int64 counters[count] (count <= FBGNN_COMM_MAX_ELEMS): staged through the
 * context's device buffer, ncclAllReduce on the context's stream, synchronises. */
int fbgnn_allreduce_counters(fbgnn_ctx *ctx, int64_t *counters, int32_t count);
/* the same for HOST doubles with FBGNN_RED_SUM / FBGNN_RED_MAX (bench.py: max over ranks of the device time) */
int fbgnn_allreduce_f64(fbgnn_ctx *ctx, double *values, int32_t count, int32_t op);
/* stream sync + a one-element all-reduce */
int fbgnn_comm_barrier(fbgnn_ctx *ctx);
int fbgnn_comm_destroy(fbgnn_ctx *ctx);

/* ---- measurement helpers ---------------------------------------------------------------- */
/* Measured MUFU (ex2.approx) throughput of the device in transcendental evaluations / s:
 * the SFU roofline denominator of SURVEY.md 8(d). */
int fbgnn_sfu_peak(fbgnn_ctx *ctx, double *evals_per_s);
/* Measured FP32 FMA issue rate (thread-instructions / s), the bound of the exact-arithmetic path */
int fbgnn_fma_peak(fbgnn_ctx *ctx, double *instr_per_s);
/* Elementwise probes of the arithmetic specification (tests): fn in {"exp","log","log1p",
 * "softplus","phi4","phi2","tanh","atanh"} (exact arithmetic), {"sfu_exp","sfu_log","sfu_softplus","sfu_phi4","sfu_phi2"}
 * "sfu_tanh","sfu_atanh" (SFU arithmetic) and the raw hardware functions {"mufu_ex2","mufu_lg2","mufu_rcp"} (tools/dump_sfu_tables.py); x,y device float32 [n]. */
int fbgnn_math_probe(fbgnn_ctx *ctx, const char *fn, const float *x, float *y, int64_t n);
/* Probe of one tcgen05.mma kind::tf32 step (M = 128, N = 16, K = 8) on `trials` operand sets: Dout = A B + Din with device
 * float32 A [T,128,8], B [T,8,16], Din / Dout [T,128,16] -- tests compare it with the integer model of csrc/fb_umma.h. */
int fbgnn_umma_probe(fbgnn_ctx *ctx, const float *A, const float *B, const float *Din, float *Dout, int32_t trials);

#ifdef __cplusplus
}
#endif
#endif /* FBGNN_H */
