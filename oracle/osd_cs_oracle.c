/* ORACLE (test infrastructure only): ordered-statistics decoding with the combination sweep (OSD-CS; Roffe et al.,
 * "Decoding across the quantum LDPC code landscape", 2020; the `ldpc` package's osd_method="osd_cs") on top of the
 * CPU oracle.  The oracle proper (fbgnn_oracle.c) is compiled into this unit, so OSD-CS reuses its sort and
 * elimination (osd0_frame), its pipelines (pipeline_frame, the BP2 frame steps) and its arithmetic unchanged.
 *
 *   orc_osd               OSD of order lam (0 = OSD-0) on a batch, the layer fbgnn_osd_decode computes
 *   orc_pipeline_osd      orc_pipeline with OSD of order lam after the last stage (cfg->osd0 is ignored)
 *   orc_bsc_pipeline_osd  orc_bsc_pipeline with OSD of order lam on the frames BP2 leaves mismatching
 *
 * Candidates T over the non-pivot columns c_0 < c_1 < ... of the reduced matrix (permuted positions, least reliable
 * first), by index: 0 the empty set (OSD-0), 1 + i the single {c_i}, then the pairs {c_i, c_j},
 * i < j < min(lam, n - rank), in lexicographic order.  T's solution is 1 on T and s'_r ^ XOR_{c in T} M[r, c] on
 * pivot piv[r]; the candidate of least (Hamming weight, index) wins. */
#include "fbgnn_oracle.c"

/* osd0_frame, then the sweep over the matrix it has reduced (M, pivots at order[n + r], inv free again);
 * e_hat holds the OSD-0 solution and is patched when a candidate is strictly lighter. */
static void osd_cs_frame(const orc_rows_t *rows, int n, int lam, const float *llr, const uint8_t *s, uint8_t *e_hat,
                         int32_t *order, int32_t *inv, uint32_t *M) {
    osd0_frame(rows, n, llr, s, e_hat, order, inv, M);
    if (lam <= 0) return;
    const int R = rows->m, W = (n + 1 + 31) / 32, RW = (R + 31) / 32;
#define OSD_BIT(r, c) ((M[(size_t)(r) * W + ((c) >> 5)] >> ((c) & 31)) & 1u)
    for (int j = 0; j < n; j++) inv[j] = 1;               /* non-pivot columns in increasing position, into inv */
    for (int r = 0; r < R; r++) inv[order[n + r]] = 0;
    int N = 0;
    for (int j = 0; j < n; j++) if (inv[j]) inv[N++] = j;
    const int lp = lam < n - R ? lam : (n - R > 0 ? n - R : 0);
    /* s' and the non-pivot columns as ceil(R/32)-word bit vectors over the rows */
    uint32_t *cv = (uint32_t *)calloc((size_t)(N + 1) * RW + 1, sizeof(uint32_t)), *sv = cv + (size_t)N * RW;
    for (int r = 0; r < R; r++) {
        sv[r >> 5] |= (uint32_t)OSD_BIT(r, n) << (r & 31);
        for (int i = 0; i < N; i++) cv[(size_t)i * RW + (r >> 5)] |= (uint32_t)OSD_BIT(r, inv[i]) << (r & 31);
    }
    int best = 0, t0 = -1, t1 = -1;
    for (int k = 0; k < RW; k++) best += __builtin_popcount(sv[k]);
    for (int i = 0; i < N; i++) {
        int w = 1;
        for (int k = 0; k < RW; k++) w += __builtin_popcount(sv[k] ^ cv[(size_t)i * RW + k]);
        if (w < best) { best = w; t0 = inv[i]; t1 = -1; }
    }
    for (int i = 0; i < lp; i++)
        for (int j = i + 1; j < lp; j++) {
            int w = 2;
            for (int k = 0; k < RW; k++)
                w += __builtin_popcount(sv[k] ^ cv[(size_t)i * RW + k] ^ cv[(size_t)j * RW + k]);
            if (w < best) { best = w; t0 = inv[i]; t1 = inv[j]; }
        }
    free(cv);
    if (t0 < 0) return;
    for (int r = 0; r < R; r++) {
        uint32_t sol = OSD_BIT(r, n) ^ OSD_BIT(r, t0);
        if (t1 >= 0) sol ^= OSD_BIT(r, t1);
        e_hat[order[order[n + r]]] = (uint8_t)sol;
    }
    e_hat[order[t0]] = 1;
    if (t1 >= 0) e_hat[order[t1]] = 1;
#undef OSD_BIT
}

/* llr [B,n], s [rank,B], e_hat [B,n] */
void orc_osd(const orc_rows_t *rows, int n, int lam, int64_t B, const float *llr, const uint8_t *s, uint8_t *e_hat) {
    const int R = rows->m, W = (n + 1 + 31) / 32;
#pragma omp parallel
    {
        int32_t *order = (int32_t *)malloc(sizeof(int32_t) * (size_t)(n + R + 1));
        int32_t *inv = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
        uint32_t *M = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)R * W + 4);
        uint8_t *sr = (uint8_t *)malloc((size_t)R + 1);
#pragma omp for schedule(dynamic, 1)
        for (int64_t b = 0; b < B; b++) {
            for (int r = 0; r < R; r++) sr[r] = s[(int64_t)r * B + b];
            osd_cs_frame(rows, n, lam, llr + b * n, sr, e_hat + b * n, order, inv, M);
        }
        free(order); free(inv); free(M); free(sr);
    }
}

/* orc_pipeline's arguments; cfg->basis_x / pivot_x / basis_z / pivot_z are required, cfg->osd0 is ignored: every
 * frame whose decision misses the syndrome after the last stage (residual syndrome non-zero) is re-solved on both
 * sides by OSD of order lam from the last stage's marginals, as pipeline_frame does for OSD-0 (bp_osd.py:135-144). */
void orc_pipeline_osd(const orc_side_t *X, const orc_side_t *Z, const orc_rows_t *lx, const orc_rows_t *lz,
                      const orc_pipe_cfg_t *cfg, int lam, const float *thr, uint64_t seed, uint64_t first_frame,
                      int64_t B, const uint8_t *noise_x, const uint8_t *noise_z, uint8_t *flags, int64_t *counters,
                      uint8_t *x_diff, uint8_t *z_diff) {
    const int n = X->n, Rx = cfg->basis_x->m, Rz = cfg->basis_z->m, Rm = Rx > Rz ? Rx : Rz;
    orc_pipe_cfg_t bp = *cfg;
    bp.osd0 = 0;
    int64_t c_flag = 0, c_blk = 0, c_s1 = 0;
    g_pipeline_early_stop = cfg->early_stop;
#pragma omp parallel reduction(+ : c_flag, c_blk, c_s1)
    {
        float *fw = (float *)malloc(sizeof(float) * pipe_float_work(X, Z, &bp));
        uint8_t *bw = (uint8_t *)malloc((size_t)(X->m + Z->m) * 2 + 8 * (size_t)n + 64);
        uint8_t *nx = (uint8_t *)malloc((size_t)n), *nz = (uint8_t *)malloc((size_t)n);
        uint8_t *xd = (uint8_t *)malloc((size_t)n), *zd = (uint8_t *)malloc((size_t)n);
        uint8_t *t = (uint8_t *)malloc((size_t)(X->m + Z->m + Rm) + 8), *sr = t + X->m + Z->m;
        uint16_t *idx = (uint16_t *)malloc(sizeof(uint16_t) * (size_t)n);
        float *ll = (float *)malloc(sizeof(float) * 2 * (size_t)n);
        int32_t *order = (int32_t *)malloc(sizeof(int32_t) * (size_t)(2 * n + Rm + 1));
        uint32_t *M = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)Rm * ((n + 32) / 32) + 4);
#pragma omp for schedule(dynamic, 1)
        for (int64_t b = 0; b < B; b++) {
            if (noise_x) { memcpy(nx, noise_x + b * n, (size_t)n); memcpy(nz, noise_z + b * n, (size_t)n); }
            else if (cfg->fixed_weight > 0) pauli_wt_frame(seed, first_frame + (uint64_t)b, n, cfg->fixed_weight, nx, nz, idx);
            else pauli_frame(seed, first_frame + (uint64_t)b, n, thr, nx, nz);
            uint8_t f = pipeline_frame(X, Z, lx, lz, &bp, nx, nz, fw, bw, xd, zd);
            if (f & 1) {
                /* pipeline_frame's work layout: the last stage's marginals L after the messages and priors; the
                 * syndromes sx, sz at the start of bw */
                const float *L = fw + X->E + Z->E + 3 * (size_t)n;
                const uint8_t *sx = bw, *sz = bw + X->m;
                float *lz_ = ll, *lx_ = ll + n;
                for (int v = 0; v < n; v++) {
                    lz_[v] = FB_SUB(fb_m_softplusf(-L[v]), fb_m_logaddexpf(-L[2 * n + v], -L[n + v]));
                    lx_[v] = FB_SUB(fb_m_softplusf(-L[2 * n + v]), fb_m_logaddexpf(-L[v], -L[n + v]));
                }
                for (int r = 0; r < Rx; r++) sr[r] = sx[cfg->pivot_x[r]];
                osd_cs_frame(cfg->basis_x, n, lam, lz_, sr, zd, order, order + n + Rm + 1, M);
                for (int r = 0; r < Rz; r++) sr[r] = sz[cfg->pivot_z[r]];
                osd_cs_frame(cfg->basis_z, n, lam, lx_, sr, xd, order, order + n + Rm + 1, M);
                for (int v = 0; v < n; v++) { xd[v] ^= nx[v]; zd[v] ^= nz[v]; }
                int flagged = 0;
                syndrome_frame(Z, xd, t);
                for (int c = 0; c < Z->m; c++) flagged |= t[c];
                syndrome_frame(X, zd, t);
                for (int c = 0; c < X->m; c++) flagged |= t[c];
                int blk = flagged | rows_any_parity(lz, xd) | rows_any_parity(lx, zd);
                f = (uint8_t)((f & ~3u) | (flagged ? 1 : 0) | (blk ? 2 : 0));
            }
            if (x_diff) memcpy(x_diff + b * n, xd, (size_t)n);
            if (z_diff) memcpy(z_diff + b * n, zd, (size_t)n);
            if (flags) flags[b] = f;
            c_flag += f & 1; c_blk += (f >> 1) & 1; c_s1 += ((f >> 2) > 0);
        }
        free(fw); free(bw); free(nx); free(nz); free(xd); free(zd); free(t); free(idx); free(ll); free(order); free(M);
    }
    if (counters) { counters[0] = B; counters[1] = c_flag; counters[2] = c_blk; counters[3] = c_s1; }
}

/* orc_bsc_pipeline with OSD of order lam on the basis osd_basis (rows osd_pivot of the pcm); BP2_OSD_Model,
 * bp_osd.py:199-274.  The frame steps are orc_bsc_pipeline's. */
void orc_bsc_pipeline_osd(const orc_side_t *S, const orc_rows_t *logical, int cn_type, int num_iter, float factor,
                          float llr_const, float p, uint64_t seed, uint64_t first_frame, int64_t B,
                          const uint8_t *noise_in, uint8_t *flags, int64_t *counters, const orc_rows_t *osd_basis,
                          const int32_t *osd_pivot, int lam) {
    const int n = S->n, m = S->m, R = osd_basis->m;
    int wd = max_cn_degree(S);
    int64_t c_flag = 0, c_blk = 0;
#pragma omp parallel reduction(+ : c_flag, c_blk)
    {
        float *msg = (float *)malloc(sizeof(float) * (size_t)(S->E + 1));
        float *work = (float *)malloc(sizeof(float) * (size_t)wd);
        float *fl = (float *)malloc(sizeof(float) * 3 * (size_t)n);
        uint8_t *by = (uint8_t *)malloc(2 * (size_t)n + 2 * (size_t)m + (size_t)R + 8);
        uint8_t *noise = by, *hard = by + n, *s = hard + n, *t = s + m, *sr = t + m;
        int32_t *order = (int32_t *)malloc(sizeof(int32_t) * (size_t)(2 * n + R + 1));
        uint32_t *M = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)R * ((n + 32) / 32) + 4);
#pragma omp for schedule(dynamic, 4)
        for (int64_t b = 0; b < B; b++) {
            if (noise_in) memcpy(noise, noise_in + b * n, (size_t)n);
            else bsc_frame(seed, first_frame + (uint64_t)b, n, p, noise);
            syndrome_frame(S, noise, s);
            for (int v = 0; v < n; v++) fl[v] = llr_const;
            bp2_frame(S, cn_type, num_iter, factor, fl, s, msg, fl + n, hard, work, fl + 2 * n);
            int mismatch = 0;
            syndrome_frame(S, hard, t);
            for (int c = 0; c < m; c++) mismatch |= (t[c] != s[c]);
            if (mismatch) {
                for (int v = 0; v < n; v++) fl[2 * n + v] = -fl[n + v];       /* llr_hat = -decoder output */
                for (int r = 0; r < R; r++) sr[r] = s[osd_pivot[r]];
                osd_cs_frame(osd_basis, n, lam, fl + 2 * n, sr, hard, order, order + n + R + 1, M);
            }
            for (int v = 0; v < n; v++) hard[v] ^= noise[v];
            int flagged = 0;
            syndrome_frame(S, hard, t);
            for (int c = 0; c < m; c++) flagged |= t[c];
            int blk = logical ? rows_any_parity(logical, hard) : flagged;
            uint8_t f = (uint8_t)((flagged ? 1 : 0) | (blk ? 2 : 0));
            if (flags) flags[b] = f;
            c_flag += f & 1; c_blk += (f >> 1) & 1;
        }
        free(msg); free(work); free(fl); free(by); free(order); free(M);
    }
    if (counters) { counters[0] = B; counters[1] = c_flag; counters[2] = c_blk; counters[3] = 0; }
}
