/*
 * oracle/eval_cpu.c -- TEST INFRASTRUCTURE, not product code.
 *
 * Plain-C restatement of the cloud-to-cloud evaluation rule of DESIGN.md section 4.7, the independent check of
 * tsar-mvs_b200/csrc/cloud_eval.cu: a brute-force double loop with no index, no pruning and no sorting.  Built with
 * -ffp-contract=off, so every float operation below is one IEEE operation in the written order.  The outer loop over
 * the query points is shared out by OpenMP; each query's minimum is taken by one thread, so the result does not depend
 * on the thread count.
 */
#include <math.h>

#include "../include/tsar_b200.h" /* TSAR_EVAL_MAX_THRESHOLDS */

static int oc_finite3(const float *p) { return isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]); }

/* dist(q, P) of the rule. */
static float oc_dist(const float *q, const float *P, long long m, float tau_max) {
    if (!oc_finite3(q)) return INFINITY;
    float best = INFINITY;
    for (long long j = 0; j < m; ++j) {
        const float *p = P + 3 * j;
        if (!oc_finite3(p)) continue;
        const float dx = p[0] - q[0], dy = p[1] - q[1], dz = p[2] - q[2];
        const float d2 = (dx * dx + dy * dy) + dz * dz;
        if (d2 < best) best = d2;
    }
    const float s = sqrtf(best);
    return s <= tau_max ? s : INFINITY;
}

static void oc_side(const float *Q, long long n, const float *P, long long m, const float *thr, int k, float tau_max,
                    long long *within, float *dist) {
#pragma omp parallel for schedule(dynamic, 16)
    for (long long i = 0; i < n; ++i) dist[i] = oc_dist(Q + 3 * i, P, m, tau_max);
    for (int t = 0; t < k; ++t) {
        long long c = 0;
        for (long long i = 0; i < n; ++i) c += dist[i] <= thr[t];
        within[t] = c;
    }
}

/* within_R / within_G: k counts each; dist_R / dist_G: n / m floats (required here). */
void oc_eval(const float *R, long long n, const float *G, long long m, const float *thr, int k, float tau_max,
             long long *within_R, long long *within_G, float *dist_R, float *dist_G) {
    oc_side(R, n, G, m, thr, k, tau_max, within_R, dist_R);
    oc_side(G, m, R, n, thr, k, tau_max, within_G, dist_G);
}
