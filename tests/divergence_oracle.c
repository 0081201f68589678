/* CPU oracle (C + OpenMP) for the divergence between two populations  --  TEST INFRASTRUCTURE ONLY.
 *
 * Input: an upper-cased byte matrix text[row*ld + site] and the row indices of two populations.  Every byte is an allele
 * (PolyFastA.py:256-258).  Per column p: Dxy_site(p) = nx*ny - sum over byte values a of cx[a]*cy[a], the number of ordered
 * pairs (i in X, j in Y) whose bytes differ.  Returns D_xy = the sum over the columns; dsite (optional) gets [L] per site. */
#include <stdint.h>
#include <string.h>

int64_t orc_divergence(const uint8_t* text, int64_t ld, int64_t L, const int32_t* rx, int64_t nx, const int32_t* ry, int64_t ny,
                       int64_t* dsite /* L or NULL */) {
    int64_t tot = 0;
#pragma omp parallel for schedule(dynamic, 16) reduction(+ : tot)
    for (int64_t p = 0; p < L; ++p) {
        int64_t cx[256], cy[256];
        memset(cx, 0, sizeof cx);
        memset(cy, 0, sizeof cy);
        for (int64_t r = 0; r < nx; ++r) cx[text[(int64_t)rx[r] * ld + p]]++;
        for (int64_t r = 0; r < ny; ++r) cy[text[(int64_t)ry[r] * ld + p]]++;
        int64_t cross = 0;
        for (int a = 0; a < 256; ++a) cross += cx[a] * cy[a];
        const int64_t d = nx * ny - cross;
        if (dsite) dsite[p] = d;
        tot += d;
    }
    return tot;
}
