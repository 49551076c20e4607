/* TEST INFRASTRUCTURE ONLY -- plain-C restatement of the feature transform behind
 * scipy.ndimage.distance_transform_edt(mask, sampling=..., return_indices=True).  The product path never links or loads
 * this file.
 *
 *  ft_oracle   for every voxel of a 3-D mask, the (z, y, x) of its nearest zero voxel as SciPy picks it: Maurer's
 *              algorithm run one line at a time, axis 0 first, then axis 1, then axis 2; before the first pass a zero voxel's
 *              feature is itself and a non-zero voxel has none (-1).  Each pass builds the stack of sites with SciPy's pop
 *              test and queries it with SciPy's comparison (a tie keeps the earlier site), every fp64 expression evaluated
 *              in SciPy's order.  Written as the general n-axis loop over a line, deliberately NOT the packed, staged
 *              form of the CUDA passes.
 *
 * Parity status: PINNED to SciPy 1.18 (tests/test_edt_ft_oracle.py: every 2x2x2 mask, random and lattice masks, with and
 * without sampling).
 *
 * Build: gcc -O2 -ffp-contract=off -shared -fPIC -o _build/libft_oracle.so ft_oracle.c
 * (-ffp-contract=off: a fused multiply-add would round differently from SciPy and change which site wins a tie)
 */
#include <stdint.h>
#include <stdlib.h>

/* one pass along axis d: ft is int32 (3, Z, Y, X), s the three spacings (1.0 each for unit spacing: exact) */
static int pass(int32_t *ft, const int64_t *shape, int d, const double *s) {
    const int64_t n = shape[0] * shape[1] * shape[2], len = shape[d];
    int64_t stride = 1;
    for (int j = 2; j > d; --j) stride *= shape[j];
    int32_t(*f)[3] = malloc((size_t)len * sizeof *f);
    int64_t *g = malloc((size_t)len * sizeof *g);
    if (!f || !g) { free(f); free(g); return -5; }
    for (int64_t start = 0; start < n; ++start) {
        int64_t coor[3] = {start / (shape[1] * shape[2]), (start / shape[2]) % shape[1], start % shape[2]};
        if (coor[d] != 0) continue; /* each line once, from its first voxel */
        for (int64_t i = 0; i < len; ++i)
            for (int j = 0; j < 3; ++j) f[i][j] = ft[j * n + start + i * stride];
        int64_t l = -1;
        for (int64_t i = 0; i < len; ++i) { /* build */
            if (f[i][0] < 0) continue;
            double wR = 0.0;
            for (int j = 0; j < 3; ++j)
                if (j != d) { double t = (double)(f[i][j] - coor[j]) * s[j]; wR += t * t; }
            while (l >= 1) {
                const int32_t *u = f[g[l - 1]], *v = f[g[l]];
                const double a = (double)(v[d] - u[d]) * s[d], b = (double)(f[i][d] - v[d]) * s[d], c = a + b;
                double uR = 0.0, vR = 0.0;
                for (int j = 0; j < 3; ++j)
                    if (j != d) {
                        const double tu = (double)(u[j] - coor[j]) * s[j], tv = (double)(v[j] - coor[j]) * s[j];
                        uR += tu * tu;
                        vR += tv * tv;
                    }
                if (c * vR - b * uR - a * wR - a * b * c <= 0.0) break;
                --l;
            }
            g[++l] = i;
        }
        if (l < 0) continue; /* no site: the line keeps what it has */
        const int64_t maxl = l;
        l = 0;
        for (int64_t i = 0; i < len; ++i) { /* query */
            double delta1 = 0.0;
            for (int j = 0; j < 3; ++j) {
                const double t = (double)(f[g[l]][j] - (j == d ? i : coor[j])) * s[j];
                delta1 += t * t;
            }
            while (l < maxl) {
                double delta2 = 0.0;
                for (int j = 0; j < 3; ++j) {
                    const double t = (double)(f[g[l + 1]][j] - (j == d ? i : coor[j])) * s[j];
                    delta2 += t * t;
                }
                if (delta1 <= delta2) break;
                delta1 = delta2;
                ++l;
            }
            for (int j = 0; j < 3; ++j) ft[j * n + start + i * stride] = f[g[l]][j];
        }
    }
    free(f);
    free(g);
    return 0;
}

/* mask: uint8 (Z, Y, X) C order, non-zero = foreground; sampling: 3 doubles or NULL; ft: int32 (3, Z, Y, X) out.
 * returns 0, or -5 when out of memory */
int ft_oracle(const uint8_t *mask, int64_t Z, int64_t Y, int64_t X, const double *sampling, int32_t *ft) {
    const int64_t shape[3] = {Z, Y, X}, n = Z * Y * X;
    const double unit[3] = {1.0, 1.0, 1.0};
    for (int64_t p = 0; p < n; ++p) {
        const int64_t c[3] = {p / (Y * X), (p / X) % Y, p % X};
        for (int j = 0; j < 3; ++j) ft[j * n + p] = mask[p] ? -1 : (int32_t)c[j];
    }
    for (int d = 0; d < 3; ++d) {
        const int rc = pass(ft, shape, d, sampling ? sampling : unit);
        if (rc) return rc;
    }
    return 0;
}
