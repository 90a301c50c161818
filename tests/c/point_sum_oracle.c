/*
 * tests/c/point_sum_oracle.c — CPU restatement of the point sum `sum(sys, f, x)` of src/core.jl:240-291.
 * TEST INFRASTRUCTURE ONLY: the checker of sphmw_point_sum (tests/point_oracle.py loads it).
 *
 * It restates the contract line by line on plain arrays, with its own cell list, and shares no code with
 * the library:
 *   cell list  create_cell_list! (core.jl:84-89): find_key of every particle, each cell's entries in
 *              DESCENDING index order (core.jl:26-41 keeps them so);
 *   home cell  find_key(x) (structs.jl:97-106): IEEE x/h, floor, minus key_phase, 1-based linear key;
 *   cells      key + key_diff[d] in the reference's order (structs.jl:70-82), only 1 <= nk <= key_max
 *              checked (core.jl:98), so face cells wrap through the linear key;
 *   accepted   dist (core.jl:8-10) r, skipped when r > sys.h (core.jl:105) — and no p == q test: a point is
 *              not a particle;
 *   sum        s = 0.0; s = s + term in traversal order; the terms 1, m*W, (m*f)*W, (m/rho)*W,
 *              ((m/rho)*f)*W, left to right; W = wendland2 (2D) | wendland3 (3D) of (sys.h, r).
 * Points outside the closed box (geometry.jl:24-30; NaN fails every comparison), and in 2D points with
 * x[3] != 0, give NaN.
 * Build: gcc -O2 -ffp-contract=off -fno-fast-math -shared -fPIC (no FMA contraction, IEEE sqrt/div).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

/* kernels.jl:108-115, :156-163 */
static double wendland2(double h, double r) {
    double x = r / h;
    if (x > 1.0) return 0.0;
    double a = (1.0 - x) * (1.0 - x);
    return 2.228169203286535 * (a * a) * (1.0 + 4.0 * x) / (h * h);
}
static double wendland3(double h, double r) {
    double x = r / h;
    if (x > 1.0) return 0.0;
    double a = (1.0 - x) * (1.0 - x);
    return 3.3422538049298023 * (a * a) * (1.0 + 4.0 * x) / (h * h * h);
}

/* box: x1_min x2_min x3_min x1_max x2_max x3_max; x: 3 x n SoA (x[3] = 0 in 2D); kind[o]: 0 count, 1 mW,
 * 2 mW*f, 3 VW, 4 VW*f; f[o]: n values (kinds 2 and 4); pts: 3 x np SoA; out[o*np + i].
 * Returns -1 if a particle is outside the box (the caller removes those first), -2 on allocation failure. */
int pso_point_sum(const double *box, double h, int64_t n, const double *x, const double *m, const double *rho,
                  int nops, const int *kind, const double *const *f, const double *pts, int64_t np, double *out) {
    int64_t phase[3], lim[3], key_max = 1, key_diff[27];
    int ndiff = 0;
    for (int a = 0; a < 3; ++a) { /* structs.jl:63-68 */
        phase[a] = (int64_t)floor(box[a] / h);
        lim[a] = (int64_t)floor(box[3 + a] / h) - phase[a] + 1;
        key_max *= lim[a];
    }
    const int dim = lim[2] == 1 ? 2 : 3;
    for (int di = -1; di <= 1; ++di)
        for (int dj = -1; dj <= 1; ++dj)
            if (dim == 2) key_diff[ndiff++] = di + lim[0] * dj;
            else
                for (int dk = -1; dk <= 1; ++dk) key_diff[ndiff++] = di + lim[0] * (dj + lim[1] * dk);

    /* the cell list: start[k-1] .. start[k] holds cell k's entries, indices descending */
    int64_t *key = (int64_t *)malloc(sizeof(int64_t) * (size_t)(n > 0 ? n : 1));
    int64_t *start = (int64_t *)calloc((size_t)key_max + 1, sizeof(int64_t));
    int64_t *entry = (int64_t *)malloc(sizeof(int64_t) * (size_t)(n > 0 ? n : 1));
    int64_t *fill = (int64_t *)malloc(sizeof(int64_t) * (size_t)key_max);
    if (!key || !start || !entry || !fill) {
        free(key); free(start); free(entry); free(fill);
        return -2;
    }
    int rc = 0;
    for (int64_t i = 0; i < n && rc == 0; ++i) {
        const double p[3] = {x[i], x[n + i], x[2 * n + i]};
        if (!(box[0] <= p[0] && p[0] <= box[3] && box[1] <= p[1] && p[1] <= box[4] && box[2] <= p[2] &&
              p[2] <= box[5])) {
            rc = -1;
            break;
        }
        key[i] = 1 + (int64_t)floor(p[0] / h) - phase[0] + lim[0] * ((int64_t)floor(p[1] / h) - phase[1]) +
                 lim[0] * lim[1] * ((int64_t)floor(p[2] / h) - phase[2]);
        start[key[i]] += 1;
    }
    if (rc == 0) {
        for (int64_t k = 1; k <= key_max; ++k) start[k] += start[k - 1];
        for (int64_t k = 0; k < key_max; ++k) fill[k] = start[k];
        for (int64_t i = n - 1; i >= 0; --i) entry[fill[key[i] - 1]++] = i; /* descending within a cell */

        for (int64_t i = 0; i < np; ++i) {
            const double q[3] = {pts[i], pts[np + i], pts[2 * np + i]};
            if (!(box[0] <= q[0] && q[0] <= box[3] && box[1] <= q[1] && q[1] <= box[4] && box[2] <= q[2] &&
                  q[2] <= box[5]) ||
                (dim == 2 && q[2] != 0.0)) {
                for (int o = 0; o < nops; ++o) out[o * np + i] = NAN;
                continue;
            }
            double s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            const int64_t k0 = 1 + (int64_t)floor(q[0] / h) - phase[0] +
                               lim[0] * ((int64_t)floor(q[1] / h) - phase[1]) +
                               lim[0] * lim[1] * ((int64_t)floor(q[2] / h) - phase[2]);
            for (int d = 0; d < ndiff; ++d) {
                const int64_t nk = k0 + key_diff[d];
                if (!(1 <= nk && nk <= key_max)) continue;
                for (int64_t e = start[nk - 1]; e < start[nk]; ++e) {
                    const int64_t j = entry[e];
                    const double dd[3] = {q[0] - x[j], q[1] - x[n + j], q[2] - x[2 * n + j]};
                    const double r = sqrt(dd[0] * dd[0] + dd[1] * dd[1] + dd[2] * dd[2]);
                    if (r > h) continue;
                    const double w = dim == 2 ? wendland2(h, r) : wendland3(h, r);
                    for (int o = 0; o < nops; ++o) {
                        double term;
                        switch (kind[o]) {
                            case 0: term = 1.0; break;
                            case 1: term = m[j] * w; break;
                            case 2: term = (m[j] * f[o][j]) * w; break;
                            case 3: term = (m[j] / rho[j]) * w; break;
                            default: term = ((m[j] / rho[j]) * f[o][j]) * w; break;
                        }
                        s[o] = s[o] + term;
                    }
                }
            }
            for (int o = 0; o < nops; ++o) out[o * np + i] = s[o];
        }
    }
    free(key); free(start); free(entry); free(fill);
    return rc;
}
