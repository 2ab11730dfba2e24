// fbgnn_lsd.cuh -- localised statistics decoding of order 0 (LSD-0; Hillmann, Berent, Quintavalle, Eisert, Wille,
// Roffe, 2024; the `ldpc` package's BpLsdDecoder): k_lsd, one CTA per frame.
//
// Specification (DESIGN.md §4 restates it).  One frame: a binary matrix H (R rows x n columns, any parity-check
// matrix), a syndrome s over its rows, reliabilities llr[v] and a sign (+1, or -1 for the binary decoder's logits).
//   Column order: ascending osd_key(sign * llr[v], v) (fbgnn_kernels.cuh) -- ties by index, -0.0 before +0.0.
//   Clusters: K = (checks C_K, columns V_K); every check of a column in V_K is in C_K; clusters share no check and no
//     column.  K is valid when s restricted to C_K lies in the GF(2) column span of H[C_K, V_K].
//   1. Start: one cluster ({c}, {}) per row c with s_c = 1; none: e = 0.
//   2. Round: for every cluster invalid at the start of the round, its candidate is the lowest-ranked column not in
//      V_K with a check in C_K.  Then, all at once, each candidate and its checks join their cluster, and clusters that
//      now share a check are united, transitively.  Validity is re-evaluated.  A valid cluster picks no candidate, but
//      a growing neighbour can absorb it.
//   3. Stop: every cluster valid -> solved (status 0).
//   4. Budget: at the start and after every round, sum |V_K| > max_cols or sum |C_K| > max_checks abandons the frame
//      (status 1); this test comes before the stop test.  An invalid cluster without a candidate abandons it with
//      status 2 (a syndrome outside H's column space).  A frame ends within max_cols + 1 rounds.
//   5. Solve: P_K = the columns of H[C_K, V_K] taken greedily in rank order while independent; x_K = the unique
//      solution supported on P_K; e = sum of the x_K (0 outside the clusters).  Row-by-row elimination with the
//      leftmost pivot (as k_osd) yields exactly P_K, so e depends only on the final clusters and the order.
// A solved frame meets its syndrome, H e = s.  An abandoned frame gets e = 0 in e_hat and keeps its bit in vbits.
//
// Implementation: the per-check slot map and the column membership bits cover the whole frame; everything else is
// indexed by slot (one per clustered check, at most max_checks) or by clustered column (at most max_cols).  Clusters
// are a union-find over slots.  Every round re-tests the clusters it changed from scratch: each such cluster's dense
// [H[C_K, V_K] | s_K] (rows x ceil((|V_K| + 1) / 32) words, packed one after another, at most max_checks x
// ceil((max_cols + 1) / 32) words in all) is eliminated by one warp.  Candidates are a per-cluster atomicMin over
// osd_key; a round's additions and unions are made by one thread, so the union-find needs no atomics.  The final
// solve ranks each cluster's columns by key and eliminates once more.
#pragma once
#include "fbgnn_kernels.cuh"

namespace fbgnn {

constexpr int LSD_MAX_COLS = 512, LSD_MAX_CHECKS = 512;            // upper limits of the budgets
constexpr int LSD_DEF_COLS = 256, LSD_DEF_CHECKS = 256;            // budget 0 = these
constexpr uint16_t LSD_NONE = 0xFFFFu;
constexpr uint8_t LSD_VALID = 1, LSD_DIRTY = 2;

struct LsdArgs {
    SideDev S;                          // graph of H
    const int *frame_list;              // optional: CTA i handles frame frame_list[i]
    View2<const float> llr;             // (b, v) reliabilities; the order key is sign * llr
    float sign;                         // +1, or -1 (binary decoder's logits)
    View2<const uint8_t> synd;          // (row, b) syndrome over H's rows
    View2<uint8_t> e_hat;               // (b, v) optional output
    uint8_t *status;                    // optional [B]: 0 solved, 1 over budget, 2 no candidate
    uint8_t *vbits;                     // optional [B][n]: a solved frame's e goes to bit `vbit` (pipeline mode)
    int vbit;
    int max_cols, max_checks;           // budgets, in [1, LSD_MAX_COLS] / [1, LSD_MAX_CHECKS]
};

// Byte offsets of the dynamic shared memory of one k_lsd CTA (host and device compute the same layout).
struct LsdLayout {
    size_t cand, moff, colkey, slot_of, vin, chk, par, rt, lrow, rowoff, nrow, ncol, cols, colrt, lcol, gcol, coloff,
        pivrow, flag, roots, M, total;
    __host__ __device__ LsdLayout(int n, int m, int MV, int MC) {
        size_t o = 0;
        auto take = [&o](size_t bytes, size_t align) { o = (o + align - 1) / align * align; size_t r = o; o += bytes; return r; };
        const size_t W = (size_t)(MV + 1 + 31) / 32;
        cand = take(8 * (size_t)MC, 8);         // u64 per slot (candidate key of the cluster rooted there)
        colkey = take(8 * (size_t)MV, 8);       // u64 per column: its key
        moff = take(4 * (size_t)MC, 4);         // u32 per root: word offset of its matrix
        nrow = take(4 * (size_t)MC, 4);         // u32 per root: |C_K|
        ncol = take(4 * (size_t)MC, 4);         // u32 per root: |V_K|
        M = take(4 * (size_t)MC * W, 4);        // u32 cluster matrices
        vin = take(4 * (size_t)((n + 31) / 32), 4);   // column membership bits
        slot_of = take(2 * (size_t)m, 2);       // u16 per check: its slot or LSD_NONE
        chk = take(2 * (size_t)MC, 2);          // u16 per slot: its check
        par = take(2 * (size_t)MC, 2);          // union-find parent
        rt = take(2 * (size_t)MC, 2);           // root of the slot this round
        lrow = take(2 * (size_t)MC, 2);         // row of the slot inside its cluster's matrix
        rowoff = take(2 * (size_t)MC, 2);       // per root: first entry of its rows in pivrow
        pivrow = take(2 * (size_t)MC, 2);       // per row of a cluster matrix: its pivot column or LSD_NONE
        roots = take(2 * (size_t)MC, 2);        // the roots of this round
        cols = take(2 * (size_t)MV, 2);         // u16 per clustered column: the column
        colrt = take(2 * (size_t)MV, 2);        // its root
        lcol = take(2 * (size_t)MV, 2);         // its column inside the cluster matrix
        gcol = take(2 * (size_t)MV, 2);         // solve: the columns grouped by cluster in rank order
        coloff = take(2 * (size_t)MC, 2);       // per root: first entry in gcol
        flag = take((size_t)MC, 1);             // per root: LSD_VALID | LSD_DIRTY
        total = (o + 15) & ~(size_t)15;
    }
};

__device__ __forceinline__ int lsd_find(const uint16_t *par, int x) {
    while (par[x] != x) x = par[x];
    return x;
}

// One warp: row-by-row elimination with the leftmost pivot of the nr x (nc + 1) matrix Mk (row stride wk words; column
// nc is s).  pivrow[r] receives row r's pivot column or LSD_NONE.  Returns whether s lies in the span of the columns.
__device__ __forceinline__ bool lsd_eliminate(uint32_t *Mk, int nr, int nc, int wk, uint16_t *pivrow, int lane) {
    const int wn = nc >> 5;
    const uint32_t last_mask = (nc & 31) ? ((1u << (nc & 31)) - 1u) : 0u;
    bool valid = true;
    for (int r = 0; r < nr; r++) {
        int p = -1;
        for (int w0 = 0; w0 <= wn && p < 0; w0 += 32) {
            const int w = w0 + lane;
            uint32_t word = w < wk ? Mk[r * wk + w] : 0u;
            if (w == wn) word &= last_mask;
            if (w > wn) word = 0u;
            const uint32_t vote = __ballot_sync(0xffffffffu, word != 0u);
            if (vote) {
                const int l = __ffs(vote) - 1;
                p = (w0 + l) * 32 + (__ffs(__shfl_sync(0xffffffffu, word, l)) - 1);
            }
        }
        if (lane == 0) pivrow[r] = p < 0 ? LSD_NONE : (uint16_t)p;
        if (p < 0) {                    // a zero row keeps its s bit from now on
            if ((Mk[r * wk + wn] >> (nc & 31)) & 1u) valid = false;
            continue;
        }
        const int pw = p >> 5;
        const uint32_t pm = 1u << (p & 31);
        __syncwarp();
        for (int i = lane; i < nr; i += 32)
            if (i != r && (Mk[i * wk + pw] & pm))
                for (int w = pw; w < wk; w++) Mk[i * wk + w] ^= Mk[r * wk + w];
        __syncwarp();
    }
    return valid;
}

// smem: LsdLayout(n, m, max_cols, max_checks)
static __global__ void __launch_bounds__(256) k_lsd(const LsdArgs a) {
    extern __shared__ __align__(16) uint8_t lsd_smem[];
    const SideDev &S = a.S;
    const int n = S.n, m = S.m, T = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = T >> 5;
    const int MV = a.max_cols, MC = a.max_checks;
    const int64_t b = a.frame_list ? a.frame_list[blockIdx.x] : blockIdx.x;
    const LsdLayout L(n, m, MV, MC);
    unsigned long long *cand = (unsigned long long *)(lsd_smem + L.cand), *colkey = (unsigned long long *)(lsd_smem + L.colkey);
    uint32_t *moff = (uint32_t *)(lsd_smem + L.moff), *nrow = (uint32_t *)(lsd_smem + L.nrow),
             *ncol = (uint32_t *)(lsd_smem + L.ncol), *M = (uint32_t *)(lsd_smem + L.M), *vin = (uint32_t *)(lsd_smem + L.vin);
    uint16_t *slot_of = (uint16_t *)(lsd_smem + L.slot_of), *chk = (uint16_t *)(lsd_smem + L.chk),
             *par = (uint16_t *)(lsd_smem + L.par), *rt = (uint16_t *)(lsd_smem + L.rt),
             *lrow = (uint16_t *)(lsd_smem + L.lrow), *rowoff = (uint16_t *)(lsd_smem + L.rowoff),
             *pivrow = (uint16_t *)(lsd_smem + L.pivrow), *roots = (uint16_t *)(lsd_smem + L.roots),
             *cols = (uint16_t *)(lsd_smem + L.cols), *colrt = (uint16_t *)(lsd_smem + L.colrt),
             *lcol = (uint16_t *)(lsd_smem + L.lcol), *gcol = (uint16_t *)(lsd_smem + L.gcol),
             *coloff = (uint16_t *)(lsd_smem + L.coloff);
    uint8_t *flag = lsd_smem + L.flag;
    __shared__ int nslots, ncols, nroots, mtotal, invalid, status;
    auto in_v = [vin](int v) { return (vin[v >> 5] >> (v & 31)) & 1u; };
    auto words = [](int nc) { return (nc + 32) >> 5; };         // ceil((nc + 1) / 32): the columns and s

    // Clear the matrices of the clusters flagged dirty and enter their rows' s bits and their columns at lcol.
    auto build = [&](int ns, int nv) {
        for (int i = tid; i < mtotal; i += T) M[i] = 0u;
        __syncthreads();
        for (int s = tid; s < ns; s += T) {
            const int r = rt[s];
            if (!(flag[r] & LSD_DIRTY) || !a.synd(chk[s], b)) continue;
            const int nc = (int)ncol[r];
            atomicOr(&M[moff[r] + lrow[s] * words(nc) + (nc >> 5)], 1u << (nc & 31));
        }
        for (int j = tid; j < nv; j += T) {
            const int r = colrt[j];
            if (!(flag[r] & LSD_DIRTY)) continue;
            const int v = cols[j], wk = words((int)ncol[r]), lc = lcol[j];
            for (int k = S.vn_ptr[v]; k < S.vn_ptr[v + 1]; k++)
                atomicOr(&M[moff[r] + lrow[slot_of[S.vn_cn[k]]] * wk + (lc >> 5)], 1u << (lc & 31));
        }
        __syncthreads();
    };

    // 1. start: a slot per check with s_c = 1
    for (int c = tid; c < m; c += T) slot_of[c] = LSD_NONE;
    for (int w = tid; w < (n + 31) / 32; w += T) vin[w] = 0u;
    if (tid == 0) { nslots = 0; ncols = 0; status = 0; }
    __syncthreads();
    for (int c = tid; c < m; c += T) {
        if (a.synd(c, b)) {
            const int s = atomicAdd(&nslots, 1);
            if (s < MC) { slot_of[c] = (uint16_t)s; chk[s] = (uint16_t)c; par[s] = (uint16_t)s; flag[s] = LSD_DIRTY; }
        }
    }
    __syncthreads();

    while (true) {
        // 4. budget
        if (nslots > MC || ncols > MV) { status = 1; break; }
        const int ns = nslots, nv = ncols;
        // the clusters: roots, per-cluster rows and columns
        for (int s = tid; s < ns; s += T) { rt[s] = (uint16_t)lsd_find(par, s); nrow[s] = 0u; ncol[s] = 0u; }
        __syncthreads();
        for (int s = tid; s < ns; s += T) lrow[s] = (uint16_t)atomicAdd(&nrow[rt[s]], 1u);
        for (int j = tid; j < nv; j += T) {
            const int r = rt[slot_of[S.vn_cn[S.vn_ptr[cols[j]]]]];
            colrt[j] = (uint16_t)r;
            lcol[j] = (uint16_t)atomicAdd(&ncol[r], 1u);
        }
        __syncthreads();
        if (tid == 0) {
            int nr = 0, ro = 0, mo = 0;
            for (int s = 0; s < ns; s++) {
                if (rt[s] != s) continue;
                roots[nr++] = (uint16_t)s;
                rowoff[s] = (uint16_t)ro;
                ro += (int)nrow[s];
                if (flag[s] & LSD_DIRTY) { moff[s] = (uint32_t)mo; mo += (int)nrow[s] * words((int)ncol[s]); }
            }
            nroots = nr; mtotal = mo; invalid = 0;
        }
        __syncthreads();
        // 2. validity of the clusters the last round changed
        build(ns, nv);
        for (int i = warp; i < nroots; i += nw) {
            const int r = roots[i];
            if (!(flag[r] & LSD_DIRTY)) continue;
            const bool ok = lsd_eliminate(M + moff[r], (int)nrow[r], (int)ncol[r], words((int)ncol[r]), pivrow + rowoff[r], lane);
            if (lane == 0) flag[r] = ok ? LSD_VALID : 0;
        }
        __syncthreads();
        for (int i = tid; i < nroots; i += T) {
            const int r = roots[i];
            flag[r] &= (uint8_t)~LSD_DIRTY;
            if (!(flag[r] & LSD_VALID)) { cand[r] = ~0ull; atomicAdd(&invalid, 1); }
        }
        __syncthreads();
        // 3. stop
        if (invalid == 0) break;
        // 2. candidates: the least key of the unclustered columns next to an invalid cluster
        for (int s = tid; s < ns; s += T) {
            const int r = rt[s], c = chk[s];
            if (flag[r] & LSD_VALID) continue;
            unsigned long long best = ~0ull;
            for (int k = S.cn_ptr[c]; k < S.cn_ptr[c + 1]; k++) {
                const int v = S.cn_vn[k];
                if (!in_v(v)) best = min(best, osd_key(a.sign * a.llr(b, v), v));
            }
            if (best != ~0ull) atomicMin(&cand[r], best);
        }
        __syncthreads();
        // additions and unions of the round, all at once (one thread)
        if (tid == 0) {
            for (int i = 0; i < nroots; i++) {
                const int r = roots[i];
                if (!(flag[r] & LSD_VALID) && cand[r] == ~0ull) status = 2;
            }
            for (int i = 0; i < nroots && !status; i++) {
                const int r = roots[i];
                if (flag[r] & LSD_VALID) continue;
                const int v = (int)(cand[r] & 0xFFFFFFFFull);
                if (!in_v(v)) {
                    vin[v >> 5] |= 1u << (v & 31);
                    const int j = ncols++;
                    if (j < MV) { cols[j] = (uint16_t)v; colkey[j] = cand[r]; }
                }
                for (int k = S.vn_ptr[v]; k < S.vn_ptr[v + 1]; k++) {
                    const int c = S.vn_cn[k];
                    const int rr = lsd_find(par, r);
                    if (slot_of[c] == LSD_NONE) {
                        const int s = nslots++;
                        if (s < MC) { slot_of[c] = (uint16_t)s; chk[s] = (uint16_t)c; par[s] = (uint16_t)rr; flag[s] = 0; }
                    } else {
                        const int q = lsd_find(par, slot_of[c]);
                        if (q != rr) par[q] = (uint16_t)rr;
                    }
                }
            }
            for (int i = 0; i < nroots && !status; i++) {
                const int r = roots[i];
                if (!(flag[r] & LSD_VALID)) flag[lsd_find(par, r)] |= LSD_DIRTY;
            }
        }
        __syncthreads();
        if (status) break;
    }

    const bool solved = status == 0;
    if (a.status && tid == 0) a.status[b] = (uint8_t)status;
    if (a.e_hat.ptr) for (int v = tid; v < n; v += T) a.e_hat(b, v) = 0;
    if (!solved) return;                                        // abandoned: e_hat = 0, vbits untouched
    if (a.vbits) for (int v = tid; v < n; v += T) a.vbits[b * n + v] &= (uint8_t)~(1u << a.vbit);

    // 5. solve: every cluster's columns in rank order, one elimination per cluster
    const int ns = nslots, nv = ncols;
    for (int j = tid; j < nv; j += T) {
        const int r = colrt[j];
        const unsigned long long k = colkey[j];
        int pos = 0;
        for (int i = 0; i < nv; i++) pos += (colrt[i] == r && colkey[i] < k);
        lcol[j] = (uint16_t)pos;
    }
    if (tid == 0) {
        int co = 0, mo = 0;
        for (int i = 0; i < nroots; i++) {
            const int r = roots[i];
            coloff[r] = (uint16_t)co; co += (int)ncol[r];
            moff[r] = (uint32_t)mo; mo += (int)nrow[r] * words((int)ncol[r]);
            flag[r] |= LSD_DIRTY;
        }
        mtotal = mo;
    }
    __syncthreads();
    for (int j = tid; j < nv; j += T) gcol[coloff[colrt[j]] + lcol[j]] = cols[j];
    build(ns, nv);
    for (int i = warp; i < nroots; i += nw) {
        const int r = roots[i], nr = (int)nrow[r], nc = (int)ncol[r], wk = words(nc);
        uint32_t *Mk = M + moff[r];
        uint16_t *pv = pivrow + rowoff[r];
        lsd_eliminate(Mk, nr, nc, wk, pv, lane);
        __syncwarp();
        for (int q = lane; q < nr; q += 32) {
            if (pv[q] == LSD_NONE || !((Mk[q * wk + (nc >> 5)] >> (nc & 31)) & 1u)) continue;
            const int v = gcol[coloff[r] + pv[q]];
            if (a.e_hat.ptr) a.e_hat(b, v) = 1;
            if (a.vbits) a.vbits[b * n + v] |= (uint8_t)(1u << a.vbit);
        }
    }
}

}  // namespace fbgnn
