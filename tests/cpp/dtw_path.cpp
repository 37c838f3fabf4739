// The DTW warping path of a pair, the checker of ss_dict_align (tests/test_align_*.py). CPU, f64, built by
// tests/align_reference.py with -ffp-contract=off like the oracle, so that mul and add stay separate IEEE operations.
//
// Spec (extension; the reference has no DTW): for La, Lb >= 1 the path is the cells (i, j) from (0, 0) to (La-1, Lb-1) in
// ascending order, found by backtracking from (La-1, Lb-1) through D as oracle/ASSUMPTIONS.h A8 defines it. At a cell other
// than (0, 0) the predecessor is the smallest D among those that exist of diag (i-1, j-1), up (i-1, j), left (i, j-1); ties
// go to the first in that order; NaN counts as +inf. The chosen value is the one fmin(fmin(up, left), diag) returned, so
// the path is a function of D's bits. An empty side, or a distance that is not finite: empty path, distance +inf.
//
// D is computed with the operations of orc_dtw (oracle/soundsym_oracle.cpp) in the same order, kept whole.
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <vector>

extern "C" {

// out_ij receives (i, j) pairs in ascending order (capacity la + lb - 1 pairs); returns the path length
size_t ref_dtw_path(const double* a, size_t la, const double* b, size_t lb, int c, uint32_t* out_ij) {
    if (la == 0 || lb == 0) return 0;
    std::vector<double> D(la * lb);
    for (size_t i = 0; i < la; i++) {
        for (size_t j = 0; j < lb; j++) {
            double cost = 0.0;
            for (int k = 0; k < c; k++) {
                const double d = a[i * c + k] - b[j * c + k];
                cost = cost + d * d;
            }
            double m;
            if (i == 0 && j == 0) m = 0.0;
            else if (i == 0) m = D[j - 1];
            else if (j == 0) m = D[(i - 1) * lb];
            else m = std::fmin(std::fmin(D[(i - 1) * lb + j], D[i * lb + j - 1]), D[(i - 1) * lb + j - 1]);
            D[i * lb + j] = cost + m;
        }
    }
    const double dist = D[la * lb - 1] / (double)(la + lb);
    if (!std::isfinite(dist)) return 0;
    std::vector<uint32_t> rev;  // (i, j) from the end
    size_t i = la - 1, j = lb - 1;
    for (;;) {
        rev.push_back((uint32_t)i);
        rev.push_back((uint32_t)j);
        if (i == 0 && j == 0) break;
        if (i == 0) {
            j--;
        } else if (j == 0) {
            i--;
        } else {
            const double up = D[(i - 1) * lb + j], left = D[i * lb + j - 1], diag = D[(i - 1) * lb + j - 1];
            const double m = std::fmin(std::fmin(up, left), diag);  // the value the recurrence added; NaN never equals it
            if (diag == m) i--, j--;
            else if (up == m) i--;
            else j--;
        }
    }
    const size_t n = rev.size() / 2;
    for (size_t s = 0; s < n; s++) {
        out_ij[2 * s] = rev[2 * (n - 1 - s)];
        out_ij[2 * s + 1] = rev[2 * (n - 1 - s) + 1];
    }
    return n;
}

}  // extern "C"
