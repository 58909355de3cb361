/*
 * Proposal-pair parse in plain C: the C twin of oracle/proposal_parse.py.  TEST INFRASTRUCTURE ONLY.
 *
 * Only tests/ and scripts/bench_proposals.py load the shared object built from this file
 * (oracle/c_proposal_parse.py -> libproposal_parse.so).  The product never links or calls it.
 *
 * It is not a restatement of reference code: the reference has no such parse.  proposal_parse.py is the
 * specification; DESIGN.md §13 lists the rule and its reconstruction points.  The per-part proposals use the
 * reference restatement's own cell arithmetic and greedy NMS, included unchanged from ppn_oracle.c, so that both
 * parsers share one definition of delta, the boxes and the suppression.
 *
 * Build with -ffp-contract=off: every operation below must round once, as numpy's do.
 */
#include "ppn_oracle.c"

/* ==== proposal-pair parse: the C twin of oracle/proposal_parse.py (NOT a reference restatement) ============
 * Per-part NMS proposals, limb scores (delta_s * limb) * delta_t of every candidate pair, and a greedy matching per
 * limb in first-reach order over the track orders (score descending, then smaller human, then smaller cell).  See
 * proposal_parse.py for the rule and DESIGN.md §13 for its reconstruction points. */

/* (limb, source, target) of every non-root part in first-reach order; returns their number, or -2 when the track
 * orders are not a tree rooted at part 0 */
int ppn_oracle_limb_tree(const ppn_oracle_geom* g, int32_t* limb, int32_t* src, int32_t* dst) {
    int n = 0;
    int32_t* how_e = (int32_t*)malloc(sizeof(int32_t) * g->K);
    int32_t* how_p = (int32_t*)malloc(sizeof(int32_t) * g->K);
    if (!how_e || !how_p) { free(how_e); free(how_p); return -1; }
    for (int k = 0; k < g->K; ++k) how_e[k] = how_p[k] = -1;
    for (int ch = 0; ch < g->n_chains; ++ch) {
        int pred = 0;
        for (int q = g->chain_off[ch]; q < g->chain_off[ch + 1]; ++q) {
            const int e = g->chain_limb[q], t = g->chain_part[q];
            if (t == 0) { n = -2; goto done; }
            if (how_e[t] < 0) { how_e[t] = e; how_p[t] = pred; limb[n] = e; src[n] = pred; dst[n] = t; ++n; }
            else if (how_e[t] != e || how_p[t] != pred) { n = -2; goto done; }
            pred = t;
        }
    }
done:
    free(how_e); free(how_p);
    return n;
}

typedef struct { float sc; int32_t i, b; } pair_t;
static int by_pair_order(const void* a, const void* b) {
    const pair_t* x = (const pair_t*)a; const pair_t* y = (const pair_t*)b;
    if (x->sc > y->sc) return -1;
    if (x->sc < y->sc) return 1;
    if (x->i != y->i) return x->i < y->i ? -1 : 1;
    return (x->b > y->b) - (x->b < y->b);
}

/* One image [C,H,W].  Output arrays hold H*W humans: root_cell[HW], part_cell[HW*K], part_score[HW*K],
 * part_box[HW*K*4]; *count = humans kept.  stats (may be NULL): [K] proposals per part, then [E] candidate pairs
 * per limb.  Returns 0, -1 (allocation) or -2 (track orders not a tree). */
int ppn_oracle_proposal_parse_image(const float* img, const ppn_oracle_geom* g, int32_t* count, int32_t* root_cell,
                                    int32_t* part_cell, float* part_score, float* part_box, int32_t* stats) {
    const int HW = g->H * g->W, K = g->K, S = g->sH * g->sW;
    int32_t tl[256], ts[256], tt[256];
    const int n_limbs = ppn_oracle_limb_tree(g, tl, ts, tt);
    if (n_limbs < 0) return n_limbs;
    int rc = -1;
    float* delta = (float*)malloc(sizeof(float) * (size_t)K * HW);
    int32_t* prop = (int32_t*)malloc(sizeof(int32_t) * (size_t)K * HW);   /* P_k: cells in NMS order */
    int32_t* n_prop = (int32_t*)calloc(K, sizeof(int32_t));
    float* cbox = (float*)malloc(sizeof(float) * 4 * HW);
    float* cscore = (float*)malloc(sizeof(float) * HW);
    int32_t* ccell = (int32_t*)malloc(sizeof(int32_t) * HW);
    int32_t* keep = (int32_t*)malloc(sizeof(int32_t) * HW);
    int32_t* cell = (int32_t*)malloc(sizeof(int32_t) * (size_t)HW * K);   /* [human][part] */
    uint8_t* used = (uint8_t*)malloc(HW);
    const size_t max_pairs = (size_t)HW * (size_t)(S < HW ? S : HW);
    pair_t* pairs = (pair_t*)malloc(sizeof(pair_t) * (max_pairs ? max_pairs : 1));
    if (!delta || !prop || !n_prop || !cbox || !cscore || !ccell || !keep || !cell || !used || !pairs) goto out;
    for (int k = 0; k < K; ++k) {
        int n = 0;
        for (int c = 0; c < HW; ++c) {
            const float d = delta_at(img, g, k, c);
            delta[(size_t)k * HW + c] = d;
            if (d > g->det_thr) { ccell[n] = c; cscore[n] = d; box_at(img, g, k, c, cbox + 4 * n); ++n; }
        }
        const int m = ppn_oracle_nms(cbox, cscore, n, g->nms_thr, 0, keep);
        if (m < 0) goto out;
        for (int j = 0; j < m; ++j) prop[(size_t)k * HW + j] = ccell[keep[j]];
        n_prop[k] = m;
    }
    const int n0 = n_prop[0];
    for (int i = 0; i < n0; ++i) {
        for (int k = 0; k < K; ++k) cell[(size_t)i * K + k] = -1;
        cell[(size_t)i * K] = prop[i];
    }
    if (stats) {
        for (int k = 0; k < K; ++k) stats[k] = n_prop[k];
        for (int e = 0; e < g->E; ++e) stats[K + e] = 0;
    }
    const float* lmb = img + (size_t)6 * K * HW;
    for (int q = 0; q < n_limbs; ++q) {
        const int e = tl[q], s = ts[q], t = tt[q];
        const int32_t* Pt = prop + (size_t)t * HW;
        size_t np = 0;
        for (int i = 0; i < n0; ++i) {
            const int a = cell[(size_t)i * K + s];
            if (a < 0) continue;
            const int ih = a / g->W, iw = a % g->W;
            const float ds = delta[(size_t)s * HW + a];
            for (int j = 0; j < n_prop[t]; ++j) {
                const int b = Pt[j], jh = b / g->W, jw = b % g->W;
                const int dy = jh - ih + g->off_h, dx = jw - iw + g->off_w;
                if (dy < 0 || dy >= g->sH || dx < 0 || dx >= g->sW) continue;
                const float lv = lmb[((size_t)(e * g->sH + dy) * g->sW + dx) * HW + a];
                const float p1 = ds * lv;
                const float sc = p1 * delta[(size_t)t * HW + b];
                if (sc > 0.0f) { pairs[np].sc = sc; pairs[np].i = i; pairs[np].b = b; ++np; }
            }
        }
        if (stats) stats[K + e] = (int32_t)np;
        qsort(pairs, np, sizeof(pair_t), by_pair_order);
        memset(used, 0, HW);
        for (size_t p = 0; p < np; ++p) {
            int32_t* ci = cell + (size_t)pairs[p].i * K;
            if (ci[t] < 0 && !used[pairs[p].b]) { ci[t] = pairs[p].b; used[pairs[p].b] = 1; }
        }
    }
    int nh = 0;
    for (int i = 0; i < n0; ++i) {
        const int32_t* ci = cell + (size_t)i * K;
        int present = 0;
        for (int k = 1; k < K; ++k) present += ci[k] >= 0;
        if (g->min_kp > present) continue;
        root_cell[nh] = ci[0];
        for (int k = 0; k < K; ++k) {
            const size_t o = (size_t)nh * K + k;
            float* bx = part_box + 4 * o;
            part_cell[o] = ci[k];
            if (ci[k] >= 0) { part_score[o] = delta[(size_t)k * HW + ci[k]]; box_at(img, g, k, ci[k], bx); }
            else { part_score[o] = 0.0f; bx[0] = bx[1] = bx[2] = bx[3] = 0.0f; }
        }
        ++nh;
    }
    *count = nh;
    rc = 0;
out:
    free(delta); free(prop); free(n_prop); free(cbox); free(cscore); free(ccell); free(keep); free(cell); free(used);
    free(pairs);
    return rc;
}

typedef struct {
    const float* head; const ppn_oracle_geom* g; int b0, b1;
    int32_t *count, *root_cell, *part_cell; float *part_score, *part_box; int32_t* stats;
    int rc;
} pjob;

static void* run_pjob(void* p) {
    pjob* j = (pjob*)p;
    const ppn_oracle_geom* g = j->g;
    const size_t HW = (size_t)g->H * g->W, K = g->K;
    const size_t per = (size_t)(6 * g->K + g->sH * g->sW * g->E) * HW;
    j->rc = 0;
    for (int b = j->b0; b < j->b1 && !j->rc; ++b)
        j->rc = ppn_oracle_proposal_parse_image(j->head + per * b, g, j->count + b, j->root_cell + HW * b,
                                                j->part_cell + HW * K * b, j->part_score + HW * K * b,
                                                j->part_box + HW * K * 4 * b,
                                                j->stats ? j->stats + (K + g->E) * (size_t)b : NULL);
    return NULL;
}

/* B images over n_threads threads (contiguous blocks); stats [B, K + E] or NULL.  Returns the first error code. */
int ppn_oracle_proposal_parse_batch(const float* head, int B, const ppn_oracle_geom* g, int n_threads, int32_t* count,
                                    int32_t* root_cell, int32_t* part_cell, float* part_score, float* part_box,
                                    int32_t* stats) {
    if (n_threads < 1) n_threads = 1;
    if (n_threads > B) n_threads = B > 0 ? B : 1;
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * n_threads);
    pjob* jobs = (pjob*)malloc(sizeof(pjob) * n_threads);
    if (!th || !jobs) { free(th); free(jobs); return -1; }
    const int per = (B + n_threads - 1) / n_threads;
    for (int t = 0; t < n_threads; ++t) {
        pjob j = { head, g, t * per, (t + 1) * per < B ? (t + 1) * per : B,
                   count, root_cell, part_cell, part_score, part_box, stats, 0 };
        if (j.b0 > B) j.b0 = B;
        jobs[t] = j;
        pthread_create(&th[t], NULL, run_pjob, &jobs[t]);
    }
    int rc = 0;
    for (int t = 0; t < n_threads; ++t) { pthread_join(th[t], NULL); if (!rc) rc = jobs[t].rc; }
    free(th); free(jobs);
    return rc;
}
