/* ORACLE (test infrastructure only): localised statistics decoding of order 0 (LSD-0; Hillmann, Berent, Quintavalle,
 * Eisert, Wille, Roffe, 2024; the `ldpc` package's BpLsdDecoder) on top of the CPU oracle.  The oracle proper
 * (fbgnn_oracle.c) is compiled into this unit, so the pipelines reuse its frame routines and arithmetic unchanged.
 *
 *   orc_lsd               LSD-0 on a batch, the layer fbgnn_lsd_decode computes
 *   orc_pipeline_lsd      orc_pipeline with LSD-0 on each side's full matrix after the last stage (cfg->osd0 ignored)
 *   orc_bsc_pipeline_lsd  orc_bsc_pipeline with LSD-0 (sign -1) on the frames BP2 leaves mismatching
 *
 * The definition (csrc/fbgnn_lsd.cuh, DESIGN.md §4), restated serially: clusters are a union-find over the checks;
 * every round takes the invalid clusters, gives each its candidate (least osd_key of an unclustered column next to
 * it), adds the candidates and their checks and unites clusters that share a check; a cluster is valid when s on its
 * checks is in the span of its columns.  Each cluster is eliminated row by row with the leftmost pivot over its
 * columns sorted by key, which both tests validity and, at the end, gives OSD-0's solution on the cluster. */
#include "fbgnn_oracle.c"

static uint64_t lsd_key(float x, int v) {
    uint32_t u;
    memcpy(&u, &x, sizeof u);
    u ^= (u >> 31) ? 0xFFFFFFFFu : 0x80000000u;               /* order-preserving float -> uint, as osd_key */
    return ((uint64_t)u << 32) | (uint32_t)v;
}

static int lsd_find(int32_t *par, int x) {
    while (par[x] != x) x = par[x];
    return x;
}

typedef struct {
    int32_t *par, *rows, *cols, *rowpos, *colpos;
    int32_t *clist, *vlist;            /* the clustered checks / columns in the order they joined */
    int nchk, ncol;
    int32_t *roots;
    uint8_t *ok;
    uint8_t *vin;
    uint64_t *key, *cand;
    uint32_t *M;
} lsd_work_t;

/* The cluster rooted at check `root`: its rows (checks, in joining order) and columns (sorted by key); eliminate
 * [H[C_K, V_K] | s_K] row by row with the leftmost pivot.  Returns validity; with e != NULL writes x_K into e. */
static int lsd_cluster(const orc_side_t *S, const uint8_t *s, int root, lsd_work_t *w, uint8_t *e) {
    const int n = S->n, m = S->m;
    int nr = 0, nc = 0;
    (void)n; (void)m;
    for (int i = 0; i < w->nchk; i++) {
        const int c = w->clist[i];
        if (lsd_find(w->par, c) == root) { w->rowpos[c] = nr; w->rows[nr++] = c; }
    }
    for (int i = 0; i < w->ncol; i++) {
        const int v = w->vlist[i];
        if (lsd_find(w->par, S->vn_cn[S->vn_ptr[v]]) == root) w->cols[nc++] = v;
    }
    for (int i = 1; i < nc; i++) {                               /* insertion sort by key */
        int v = w->cols[i], j = i;
        while (j > 0 && w->key[w->cols[j - 1]] > w->key[v]) { w->cols[j] = w->cols[j - 1]; j--; }
        w->cols[j] = v;
    }
    const int W = (nc + 1 + 31) / 32;
    uint32_t *M = w->M;
    memset(M, 0, sizeof(uint32_t) * (size_t)nr * W);
    for (int j = 0; j < nc; j++) {
        const int v = w->cols[j];
        for (int k = S->vn_ptr[v]; k < S->vn_ptr[v + 1]; k++)
            M[(size_t)w->rowpos[S->vn_cn[k]] * W + (j >> 5)] |= 1u << (j & 31);
    }
    for (int r = 0; r < nr; r++)
        if (s[w->rows[r]]) M[(size_t)r * W + (nc >> 5)] |= 1u << (nc & 31);
#define LSD_BIT(r, j) ((M[(size_t)(r) * W + ((j) >> 5)] >> ((j) & 31)) & 1u)
    int valid = 1;
    for (int r = 0; r < nr; r++) {
        int p = -1;
        for (int j = 0; j < nc; j++) if (LSD_BIT(r, j)) { p = j; break; }
        w->colpos[r] = p;
        if (p < 0) { if (LSD_BIT(r, nc)) valid = 0; continue; }
        for (int i = 0; i < nr; i++)
            if (i != r && LSD_BIT(i, p))
                for (int q = 0; q < W; q++) M[(size_t)i * W + q] ^= M[(size_t)r * W + q];
    }
    if (e)
        for (int r = 0; r < nr; r++)
            if (w->colpos[r] >= 0 && LSD_BIT(r, nc)) e[w->cols[w->colpos[r]]] = 1;
#undef LSD_BIT
    return valid;
}

/* One frame of LSD-0 on S (rows = checks).  Returns the status: 0 solved, 1 over budget, 2 no candidate.  e_hat is
 * written only when the frame is solved. */
static int lsd_frame(const orc_side_t *S, int max_cols, int max_checks, float sign, const float *llr, const uint8_t *s,
                     uint8_t *e_hat, lsd_work_t *w) {
    const int n = S->n, m = S->m;
    int32_t *roots = w->roots;
    uint8_t *ok = w->ok;
    w->nchk = w->ncol = 0;
    for (int v = 0; v < n; v++) { w->vin[v] = 0; w->key[v] = lsd_key(sign * llr[v], v); }
    for (int c = 0; c < m; c++) {
        w->par[c] = s[c] ? c : -1;
        if (s[c]) w->clist[w->nchk++] = c;
    }
    int status;
    for (;;) {
        if (w->ncol > max_cols || w->nchk > max_checks) { status = 1; break; }
        int nr = 0, invalid = 0;
        for (int i = 0; i < w->nchk; i++) if (w->par[w->clist[i]] == w->clist[i]) roots[nr++] = w->clist[i];
        for (int i = 0; i < nr; i++) {
            ok[i] = (uint8_t)lsd_cluster(S, s, roots[i], w, NULL);
            invalid += !ok[i];
        }
        if (!invalid) {
            memset(e_hat, 0, (size_t)n);
            for (int i = 0; i < nr; i++) lsd_cluster(S, s, roots[i], w, e_hat);
            status = 0;
            break;
        }
        for (int i = 0; i < nr; i++) w->cand[roots[i]] = ~(uint64_t)0;
        for (int q = 0; q < w->nchk; q++) {
            const int c = w->clist[q], r = lsd_find(w->par, c);
            int i = 0;
            while (roots[i] != r) i++;
            if (ok[i]) continue;
            for (int k = S->cn_ptr[c]; k < S->cn_ptr[c + 1]; k++) {
                const int v = S->cn_vn[k];
                if (!w->vin[v] && w->key[v] < w->cand[r]) w->cand[r] = w->key[v];
            }
        }
        status = 0;
        for (int i = 0; i < nr; i++) if (!ok[i] && w->cand[roots[i]] == ~(uint64_t)0) status = 2;
        if (status) break;
        for (int i = 0; i < nr; i++) {
            if (ok[i]) continue;
            const int r = roots[i], v = (int)(w->cand[r] & 0xFFFFFFFFu);
            if (!w->vin[v]) { w->vin[v] = 1; w->vlist[w->ncol++] = v; }
            for (int k = S->vn_ptr[v]; k < S->vn_ptr[v + 1]; k++) {
                const int c = S->vn_cn[k], rr = lsd_find(w->par, r);
                if (w->par[c] < 0) { w->par[c] = rr; w->clist[w->nchk++] = c; }
                else {
                    const int q = lsd_find(w->par, c);
                    if (q != rr) w->par[q] = rr;
                }
            }
        }
    }
    return status;
}

static void lsd_work_alloc(lsd_work_t *w, int n, int m, int max_cols) {
    const int W = (max_cols + 2 + 31) / 32;
    w->par = (int32_t *)malloc(sizeof(int32_t) * (size_t)m + 4);
    w->rows = (int32_t *)malloc(sizeof(int32_t) * (size_t)m + 4);
    w->rowpos = (int32_t *)malloc(sizeof(int32_t) * (size_t)m + 4);
    w->colpos = (int32_t *)malloc(sizeof(int32_t) * (size_t)m + 4);
    w->cols = (int32_t *)malloc(sizeof(int32_t) * (size_t)n + 4);
    w->vin = (uint8_t *)malloc((size_t)n + 4);
    w->key = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)n + 8);
    w->cand = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)m + 8);
    w->M = (uint32_t *)malloc(sizeof(uint32_t) * ((size_t)m * W + 4));
    w->clist = (int32_t *)malloc(sizeof(int32_t) * (size_t)m + 4);
    w->vlist = (int32_t *)malloc(sizeof(int32_t) * (size_t)n + 4);
    w->roots = (int32_t *)malloc(sizeof(int32_t) * (size_t)m + 4);
    w->ok = (uint8_t *)malloc((size_t)m + 4);
}

static void lsd_work_free(lsd_work_t *w) {
    free(w->par); free(w->rows); free(w->rowpos); free(w->colpos); free(w->cols); free(w->vin); free(w->key);
    free(w->cand); free(w->M); free(w->clist); free(w->vlist); free(w->roots); free(w->ok);
}

/* llr [B,n], s [m,B] (all rows of S), e_hat [B,n] (0 where abandoned), status [B] (optional) */
void orc_lsd(const orc_side_t *S, int max_cols, int max_checks, int64_t B, const float *llr, const uint8_t *s,
             uint8_t *e_hat, uint8_t *status) {
    const int n = S->n, m = S->m;
#pragma omp parallel
    {
        lsd_work_t w;
        lsd_work_alloc(&w, n, m, max_cols);
        uint8_t *sr = (uint8_t *)malloc((size_t)m + 1);
#pragma omp for schedule(dynamic, 1)
        for (int64_t b = 0; b < B; b++) {
            for (int c = 0; c < m; c++) sr[c] = s[(int64_t)c * B + b];
            int st = lsd_frame(S, max_cols, max_checks, 1.0f, llr + b * n, sr, e_hat + b * n, &w);
            if (st) memset(e_hat + b * n, 0, (size_t)n);
            if (status) status[b] = (uint8_t)st;
        }
        free(sr);
        lsd_work_free(&w);
    }
}

/* orc_pipeline's arguments (cfg->osd0 and the bases are ignored): every frame whose decision misses the syndrome after
 * the last stage is re-solved on both sides by LSD-0 from the last stage's marginals -- hx with osd_llrz and syndrome_x,
 * hz with osd_llrx and syndrome_z, the LLRs of orc_pipeline_osd (bp_osd.py:135-144); a side LSD-0 abandons keeps its BP
 * decision.  unsolved (optional [B]): 1 where a side whose decision missed its syndrome was abandoned. */
void orc_pipeline_lsd(const orc_side_t *X, const orc_side_t *Z, const orc_rows_t *lx, const orc_rows_t *lz,
                      const orc_pipe_cfg_t *cfg, int max_cols, int max_checks, const float *thr, uint64_t seed,
                      uint64_t first_frame, int64_t B, const uint8_t *noise_x, const uint8_t *noise_z, uint8_t *flags,
                      int64_t *counters, uint8_t *x_diff, uint8_t *z_diff, uint8_t *unsolved) {
    const int n = X->n, Mm = X->m > Z->m ? X->m : Z->m;
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
        uint8_t *t = (uint8_t *)malloc((size_t)Mm + 8);
        uint16_t *idx = (uint16_t *)malloc(sizeof(uint16_t) * (size_t)n);
        float *ll = (float *)malloc(sizeof(float) * 2 * (size_t)n);
        lsd_work_t lw;
        lsd_work_alloc(&lw, n, Mm, max_cols);
#pragma omp for schedule(dynamic, 1)
        for (int64_t b = 0; b < B; b++) {
            if (noise_x) { memcpy(nx, noise_x + b * n, (size_t)n); memcpy(nz, noise_z + b * n, (size_t)n); }
            else if (cfg->fixed_weight > 0) pauli_wt_frame(seed, first_frame + (uint64_t)b, n, cfg->fixed_weight, nx, nz, idx);
            else pauli_frame(seed, first_frame + (uint64_t)b, n, thr, nx, nz);
            uint8_t f = pipeline_frame(X, Z, lx, lz, &bp, nx, nz, fw, bw, xd, zd);
            int left = 0;
            if (f & 1) {
                /* pipeline_frame's work layout: the last stage's marginals L after the messages and priors; the
                 * syndromes sx, sz at the start of bw; xd / zd hold x_hat ^ noise_x / z_hat ^ noise_z */
                const float *L = fw + X->E + Z->E + 3 * (size_t)n;
                const uint8_t *sx = bw, *sz = bw + X->m;
                float *lz_ = ll, *lx_ = ll + n;
                for (int v = 0; v < n; v++) {
                    lz_[v] = FB_SUB(fb_m_softplusf(-L[v]), fb_m_logaddexpf(-L[2 * n + v], -L[n + v]));
                    lx_[v] = FB_SUB(fb_m_softplusf(-L[2 * n + v]), fb_m_logaddexpf(-L[v], -L[n + v]));
                }
                for (int v = 0; v < n; v++) { xd[v] ^= nx[v]; zd[v] ^= nz[v]; }          /* back to x_hat, z_hat */
                int miss_z = 0, miss_x = 0;
                syndrome_frame(X, zd, t);
                for (int c = 0; c < X->m; c++) miss_z |= t[c] != sx[c];
                syndrome_frame(Z, xd, t);
                for (int c = 0; c < Z->m; c++) miss_x |= t[c] != sz[c];
                if (lsd_frame(X, max_cols, max_checks, 1.0f, lz_, sx, zd, &lw)) left |= miss_z;
                if (lsd_frame(Z, max_cols, max_checks, 1.0f, lx_, sz, xd, &lw)) left |= miss_x;
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
            if (unsolved) unsolved[b] = (uint8_t)left;
            c_flag += f & 1; c_blk += (f >> 1) & 1; c_s1 += ((f >> 2) > 0);
        }
        free(fw); free(bw); free(nx); free(nz); free(xd); free(zd); free(t); free(idx); free(ll);
        lsd_work_free(&lw);
    }
    if (counters) { counters[0] = B; counters[1] = c_flag; counters[2] = c_blk; counters[3] = c_s1; }
}

/* orc_bsc_pipeline with LSD-0 on S itself (sign -1: llr_hat = -decoder output) for the frames BP2 leaves mismatching;
 * BP2_OSD_Model with an LSD decoder.  unsolved (optional [B]): 1 where LSD-0 abandoned the frame. */
void orc_bsc_pipeline_lsd(const orc_side_t *S, const orc_rows_t *logical, int cn_type, int num_iter, float factor,
                          float llr_const, float p, uint64_t seed, uint64_t first_frame, int64_t B,
                          const uint8_t *noise_in, uint8_t *flags, int64_t *counters, int max_cols, int max_checks,
                          uint8_t *unsolved) {
    const int n = S->n, m = S->m;
    int wd = max_cn_degree(S);
    int64_t c_flag = 0, c_blk = 0;
#pragma omp parallel reduction(+ : c_flag, c_blk)
    {
        float *msg = (float *)malloc(sizeof(float) * (size_t)(S->E + 1));
        float *work = (float *)malloc(sizeof(float) * (size_t)wd);
        float *fl = (float *)malloc(sizeof(float) * 3 * (size_t)n);
        uint8_t *by = (uint8_t *)malloc(2 * (size_t)n + 2 * (size_t)m + 8);
        uint8_t *noise = by, *hard = by + n, *s = hard + n, *t = s + m;
        lsd_work_t lw;
        lsd_work_alloc(&lw, n, m, max_cols);
#pragma omp for schedule(dynamic, 4)
        for (int64_t b = 0; b < B; b++) {
            if (noise_in) memcpy(noise, noise_in + b * n, (size_t)n);
            else bsc_frame(seed, first_frame + (uint64_t)b, n, p, noise);
            syndrome_frame(S, noise, s);
            for (int v = 0; v < n; v++) fl[v] = llr_const;
            bp2_frame(S, cn_type, num_iter, factor, fl, s, msg, fl + n, hard, work, fl + 2 * n);
            int mismatch = 0, left = 0;
            syndrome_frame(S, hard, t);
            for (int c = 0; c < m; c++) mismatch |= (t[c] != s[c]);
            if (mismatch) left = lsd_frame(S, max_cols, max_checks, -1.0f, fl + n, s, hard, &lw) != 0;
            for (int v = 0; v < n; v++) hard[v] ^= noise[v];
            int flagged = 0;
            syndrome_frame(S, hard, t);
            for (int c = 0; c < m; c++) flagged |= t[c];
            int blk = logical ? rows_any_parity(logical, hard) : flagged;
            uint8_t f = (uint8_t)((flagged ? 1 : 0) | (blk ? 2 : 0));
            if (flags) flags[b] = f;
            if (unsolved) unsolved[b] = (uint8_t)left;
            c_flag += f & 1; c_blk += (f >> 1) & 1;
        }
        free(msg); free(work); free(fl); free(by);
        lsd_work_free(&lw);
    }
    if (counters) { counters[0] = B; counters[1] = c_flag; counters[2] = c_blk; counters[3] = 0; }
}
