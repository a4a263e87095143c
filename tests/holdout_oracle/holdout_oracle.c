/*
 * tests/holdout_oracle/holdout_oracle.c — CPU restatement of the MASKED BigCLAM step (held-out pairs, DESIGN.md (f) f-5)
 * and of the held-out log-likelihood.
 *
 * TEST INFRASTRUCTURE ONLY, like oracle/bigclam_oracle.c, whose arithmetic it extends: the helpers below are the same
 * statements in the same order and built with the same flags (holdout_oracle.py), so with empty held-out lists
 * oracle_step_masked gives the same bits as oracle_step.
 *
 * The masked objective leaves every held-out pair (u, v) out of the edge term AND the non-edge term.  sumF keeps its
 * meaning (column sums of all of F), so in the per-node form of bigclam4-7.scala:157-181 a held-out pair is an extra
 * "edge" whose term is x_uv itself and whose weight is 1:
 *
 *   llh_u   = sum_{v in N(u)} (log(1 - p_uv) + x_uv) + sum_{v in HO(u)} x_uv - fu.sumF + fu.fu
 *   grad_u  = sum_{v in N(u)} fv / (1 - p_uv)        + sum_{v in HO(u)} fv   - sumF    + fu
 *   llh'(s) = sum_{v in N(u)} T(nf.fv)               + sum_{v in HO(u)} nf.fv - nf.((sumF - fu) + nf) + nf.nf
 *
 * Every sum over a node's pairs is ONE left fold in list order: the neighbour list first, then the held-out list.
 * Held-out log-likelihood (each pair once, u < v, nodes in order, pairs in list order):
 *   L_HO = sum_{held-out edges} log(1 - p) + sum_{held-out non-edges} log(p),  p = clamp(exp(-x), MIN_P_, MAX_P_) (:166).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

typedef struct {   /* == oracle_params (oracle/bigclam_oracle.c) */
    int32_t k;
    int32_t max_inter;
    double alpha;
    double beta;
    double min_p;
    double max_p;
    double min_f;
    double max_f;
} oracle_params;

static void step_sizes(double beta, int32_t max_inter, double *out) {
    double s = 1.0;
    out[0] = s;
    for (int i = 1; i <= max_inter; ++i) { s *= beta; out[i] = s; }
}

static inline double dot_seq(const double *a, const double *b, int k) {
    double acc = 0.0;
    for (int i = 0; i < k; ++i) acc += a[i] * b[i];
    return acc;
}

static inline double edge_term(double x, const oracle_params *p, double *one_minus_p) {
    double pr = fmin(fmax(exp(-x), p->min_p), p->max_p);
    if (one_minus_p) *one_minus_p = 1.0 - pr;
    return log(1.0 - pr) + x;
}

/* PRE block over N(u) then HO(u).  Returns llh_u, writes grad (k). */
static double pre_node(const int64_t *rowptr, const int32_t *col, const int64_t *ho_rowptr, const int32_t *ho_col, int64_t u,
                       const double *F, const double *sumF, const oracle_params *p, double *grad) {
    const int k = p->k;
    const double *fu = F + (size_t)u * k;
    double fusfT = dot_seq(fu, sumF, k);
    double fufuT = dot_seq(fu, fu, k);
    double s1 = 0.0;
    for (int i = 0; i < k; ++i) grad[i] = 0.0;
    int first = 1;
    for (int64_t e = rowptr[u]; e < rowptr[u + 1]; ++e) {
        const double *fv = F + (size_t)col[e] * k;
        double x = dot_seq(fu, fv, k);
        double omp_;
        double t = edge_term(x, p, &omp_);
        double w = 1.0 / omp_;
        if (first) {
            s1 = t;
            for (int i = 0; i < k; ++i) grad[i] = fv[i] * w;
            first = 0;
        } else {
            s1 = s1 + t;
            for (int i = 0; i < k; ++i) grad[i] = grad[i] + fv[i] * w;
        }
    }
    for (int64_t e = ho_rowptr[u]; e < ho_rowptr[u + 1]; ++e) {      /* held-out pairs: term x, weight 1 */
        const double *fv = F + (size_t)ho_col[e] * k;
        double x = dot_seq(fu, fv, k);
        if (first) {
            s1 = x;
            for (int i = 0; i < k; ++i) grad[i] = fv[i];
            first = 0;
        } else {
            s1 = s1 + x;
            for (int i = 0; i < k; ++i) grad[i] = grad[i] + fv[i];
        }
    }
    for (int i = 0; i < k; ++i) grad[i] = (grad[i] - sumF[i]) + fu[i];
    return (s1 - fusfT) + fufuT;
}

static double *g_margin_out = NULL;
#ifdef _OPENMP
#pragma omp threadprivate(g_margin_out)
#endif

static int ls_trial(const int64_t *rowptr, const int32_t *col, const int64_t *ho_rowptr, const int32_t *ho_col, int64_t u,
                    const double *F, const double *sumF, const oracle_params *p,
                    const double *grad, double llh_u, double s, double *newfu, double *sfT) {
    const int k = p->k;
    const double *fu = F + (size_t)u * k;
    for (int i = 0; i < k; ++i) {
        double x = fu[i] + s * grad[i];
        newfu[i] = fmin(fmax(x, p->min_f), p->max_f);
    }
    for (int i = 0; i < k; ++i) sfT[i] = (sumF[i] - fu[i]) + newfu[i];
    double acc = 0.0;
    int first = 1;
    for (int64_t e = rowptr[u]; e < rowptr[u + 1]; ++e) {
        const double *fv = F + (size_t)col[e] * k;
        double xc = dot_seq(newfu, fv, k);
        double t = edge_term(xc, p, NULL);
        if (first) { acc = t; first = 0; } else acc = acc + t;
    }
    for (int64_t e = ho_rowptr[u]; e < ho_rowptr[u + 1]; ++e) {
        const double *fv = F + (size_t)ho_col[e] * k;
        double xc = dot_seq(newfu, fv, k);
        if (first) { acc = xc; first = 0; } else acc = acc + xc;
    }
    double result = (acc - dot_seq(newfu, sfT, k)) + dot_seq(newfu, newfu, k);
    double as = p->alpha * s;
    double arm = 0.0;
    for (int i = 0; i < k; ++i) arm += (as * grad[i]) * grad[i];
    if (g_margin_out) *g_margin_out = result - (llh_u + arm);
    return result >= (llh_u + arm);
}

/* Armijo margins llh'(s_j) - (llh_u + alpha s_j |g|^2) of all candidates of the given nodes, and their llh_u (tie proofs). */
void oracle_armijo_margins_masked(int64_t n, const int64_t *rowptr, const int32_t *col, const int64_t *ho_rowptr, const int32_t *ho_col,
                                  const oracle_params *p, const double *F, const double *sumF, const int64_t *nodes, int64_t count,
                                  double *margins_out, double *llh_u_out) {
    (void)n;
    const int k = p->k;
    const int nsteps = p->max_inter + 1;
    double *steps = (double *)malloc(sizeof(double) * (size_t)nsteps);
    step_sizes(p->beta, p->max_inter, steps);
    double *grad = (double *)malloc(sizeof(double) * (size_t)k * 3);
    double *newfu = grad + k, *sfT = grad + 2 * (size_t)k;
    for (int64_t i = 0; i < count; ++i) {
        const int64_t u = nodes[i];
        const double llh_u = pre_node(rowptr, col, ho_rowptr, ho_col, u, F, sumF, p, grad);
        llh_u_out[i] = llh_u;
        for (int j = 0; j < nsteps; ++j) {
            double m = 0.0;
            g_margin_out = &m;
            (void)ls_trial(rowptr, col, ho_rowptr, ho_col, u, F, sumF, p, grad, llh_u, steps[j], newfu, sfT);
            g_margin_out = NULL;
            margins_out[i * nsteps + j] = m;
        }
    }
    free(grad);
    free(steps);
}

static double llh_node(const int64_t *rowptr, const int32_t *col, const int64_t *ho_rowptr, const int32_t *ho_col, int64_t u,
                       const double *F, const double *sumF, const oracle_params *p) {
    const int k = p->k;
    const double *fu = F + (size_t)u * k;
    double fusfT = dot_seq(fu, sumF, k);
    double fufuT = dot_seq(fu, fu, k);
    double acc = 0.0;
    int first = 1;
    for (int64_t e = rowptr[u]; e < rowptr[u + 1]; ++e) {
        const double *fv = F + (size_t)col[e] * k;
        double x = dot_seq(fu, fv, k);
        double t = edge_term(x, p, NULL);
        if (first) { acc = t; first = 0; } else acc = acc + t;
    }
    for (int64_t e = ho_rowptr[u]; e < ho_rowptr[u + 1]; ++e) {
        const double *fv = F + (size_t)ho_col[e] * k;
        double x = dot_seq(fu, fv, k);
        if (first) { acc = x; first = 0; } else acc = acc + x;
    }
    return (acc - fusfT) + fufuT;
}

/* Masked LLH = sum_u llh_node(u) in node order. */
double oracle_llh_masked(int64_t n, const int64_t *rowptr, const int32_t *col, const int64_t *ho_rowptr, const int32_t *ho_col,
                         const oracle_params *p, const double *F, const double *sumF, double *per_node) {
    double *tmp = per_node ? per_node : (double *)malloc(sizeof(double) * (size_t)n);
#pragma omp parallel for schedule(dynamic, 256)
    for (int64_t u = 0; u < n; ++u) tmp[u] = llh_node(rowptr, col, ho_rowptr, ho_col, u, F, sumF, p);
    double llh = 0.0;
    for (int64_t u = 0; u < n; ++u) llh += tmp[u];
    if (!per_node) free(tmp);
    return llh;
}

/* One masked backtrackingLineSearchs call; arguments as oracle_step (oracle/bigclam_oracle.c) plus the held-out lists. */
double oracle_step_masked(int64_t n, const int64_t *rowptr, const int32_t *col, const int64_t *ho_rowptr, const int32_t *ho_col,
                          const oracle_params *p, const double *F_in, double *sumF,
                          const uint8_t *node_mask, double *F_out,
                          int64_t *n_updated_out, int8_t *accepted, int8_t *trials_out,
                          int32_t early_exit, double *grad_out, double *llh_u_out) {
    const int k = p->k;
    const int nsteps = p->max_inter + 1;
    double *steps = (double *)malloc(sizeof(double) * (size_t)nsteps);
    step_sizes(p->beta, p->max_inter, steps);
    int8_t *acc_idx = accepted ? accepted : (int8_t *)malloc((size_t)n);

#pragma omp parallel
    {
        double *grad = (double *)malloc(sizeof(double) * (size_t)k * 4);
        double *newfu = grad + k, *sfT = grad + 2 * (size_t)k, *best = grad + 3 * (size_t)k;
#pragma omp for schedule(dynamic, 64)
        for (int64_t u = 0; u < n; ++u) {
            const double *fu = F_in + (size_t)u * k;
            double *out = F_out + (size_t)u * k;
            int8_t chosen = -1, ntr = 0;
            int in_uset = (node_mask == NULL) || node_mask[u];
            if (in_uset && rowptr[u + 1] > rowptr[u]) {               /* an empty NEIGHBOUR list: never updated */
                double llh_u = pre_node(rowptr, col, ho_rowptr, ho_col, u, F_in, sumF, p, grad);
                if (grad_out) memcpy(grad_out + (size_t)u * k, grad, sizeof(double) * (size_t)k);
                if (llh_u_out) llh_u_out[u] = llh_u;
                for (int j = 0; j < nsteps; ++j) {
                    ++ntr;
                    int pass = ls_trial(rowptr, col, ho_rowptr, ho_col, u, F_in, sumF, p, grad, llh_u, steps[j], newfu, sfT);
                    if (pass && chosen < 0) {
                        chosen = (int8_t)j;
                        memcpy(best, newfu, sizeof(double) * (size_t)k);
                        if (early_exit) break;
                    }
                }
            } else {
                if (grad_out) memset(grad_out + (size_t)u * k, 0, sizeof(double) * (size_t)k);
                if (llh_u_out) llh_u_out[u] = llh_node(rowptr, col, ho_rowptr, ho_col, u, F_in, sumF, p);
            }
            acc_idx[u] = chosen;
            if (trials_out) trials_out[u] = ntr;
            memcpy(out, chosen >= 0 ? best : fu, sizeof(double) * (size_t)k);
        }
        free(grad);
    }

    int64_t n_upd = 0;
    double *A = (double *)calloc((size_t)k * 2, sizeof(double));
    double *B = A + k;
    for (int64_t u = 0; u < n; ++u) {
        if (acc_idx[u] < 0) continue;
        const double *o = F_in + (size_t)u * k, *nw = F_out + (size_t)u * k;
        if (n_upd == 0) { for (int i = 0; i < k; ++i) { A[i] = o[i]; B[i] = nw[i]; } }
        else            { for (int i = 0; i < k; ++i) { A[i] = A[i] + o[i]; B[i] = B[i] + nw[i]; } }
        ++n_upd;
    }
    if (n_upd > 0) for (int i = 0; i < k; ++i) sumF[i] = sumF[i] - (A[i] - B[i]);
    free(A);
    if (n_updated_out) *n_updated_out = n_upd;
    if (!accepted) free(acc_idx);
    free(steps);

    return oracle_llh_masked(n, rowptr, col, ho_rowptr, ho_col, p, F_out, sumF, NULL);
}

/* SGDFindC (variant 4, bigclam4-7.scala:225-243) on the masked objective; as oracle_run. */
int64_t oracle_run_masked(int64_t n, const int64_t *rowptr, const int32_t *col, const int64_t *ho_rowptr, const int32_t *ho_col,
                          const oracle_params *p, double *F, double *sumF, double rel_tol, int64_t max_outer,
                          double *llh_out, double *llh_trace, int64_t trace_cap) {
    const size_t bytes = sizeof(double) * (size_t)n * (size_t)p->k;
    double *Fb = (double *)malloc(bytes);
    int64_t calls = 0;
    double LLHold = oracle_step_masked(n, rowptr, col, ho_rowptr, ho_col, p, F, sumF, NULL, Fb, NULL, NULL, NULL, 1, NULL, NULL);
    memcpy(F, Fb, bytes);
    if (llh_trace && calls < trace_cap) llh_trace[calls] = LLHold;
    ++calls;
    while (max_outer == 0 || calls < max_outer) {
        double newLLH = oracle_step_masked(n, rowptr, col, ho_rowptr, ho_col, p, F, sumF, NULL, Fb, NULL, NULL, NULL, 1, NULL, NULL);
        memcpy(F, Fb, bytes);
        if (llh_trace && calls < trace_cap) llh_trace[calls] = newLLH;
        ++calls;
        if (fabs(1.0 - newLLH / LLHold) < rel_tol) break;
        LLHold = newLLH;
    }
    free(Fb);
    if (llh_out) *llh_out = LLHold;
    return calls;
}

/* L_HO over the pairs (u, v), v > u, nodes in order, pairs in list order. */
double oracle_holdout_llh(int64_t n, const int64_t *ho_rowptr, const int32_t *ho_col, const uint8_t *ho_is_edge,
                          const oracle_params *p, const double *F, int64_t *n_pairs_out) {
    const int k = p->k;
    double acc = 0.0;
    int64_t pairs = 0;
    for (int64_t u = 0; u < n; ++u) {
        const double *fu = F + (size_t)u * k;
        for (int64_t e = ho_rowptr[u]; e < ho_rowptr[u + 1]; ++e) {
            const int64_t v = ho_col[e];
            if (v <= u) continue;
            double x = dot_seq(fu, F + (size_t)v * k, k);
            double pr = fmin(fmax(exp(-x), p->min_p), p->max_p);
            acc += ho_is_edge[e] ? log(1.0 - pr) : log(pr);
            ++pairs;
        }
    }
    if (n_pairs_out) *n_pairs_out = pairs;
    return acc;
}
