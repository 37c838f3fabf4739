// DTW with a Sakoe-Chiba band: the checker of ss_dict_set_dtw_band (tests/test_band_*.py). CPU, f64, built by
// tests/band_reference.py with -ffp-contract=off like the oracle, so that mul and add stay separate IEEE operations.
//
// Spec (A10, DESIGN.md §3.1f; extends oracle/ASSUMPTIONS.h A8). The radius r is a non-negative integer; r = 0 means no band.
// For r >= 1, cell (i, j) of a pair of lengths (La, Lb) is inside the band iff
//     |i (Lb - 1) - j (La - 1)| <= r max(La - 1, Lb - 1)        (64-bit integers)
// A cell outside the band has D = +inf and is never a predecessor, exactly like the missing neighbours of row 0 and column 0.
// Inside it, the recurrence, its operation order, the normalisation D(La-1, Lb-1) / (La + Lb), the (distance, index) order
// of the top-k and the NaN rule are A8's. The warping path is the backtrack of tests/cpp/dtw_path.cpp through the banded D.
//
// D is computed with the operations of orc_dtw (oracle/soundsym_oracle.cpp) in the same order; r = 0 is orc_dtw itself.
// Local costs of cells outside the band are not computed (they cannot reach D).
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <limits>
#include <thread>
#include <utility>
#include <vector>

namespace {

constexpr double kInf = std::numeric_limits<double>::infinity();

// the full banded matrix D (la x lb, la, lb >= 1)
void band_matrix(const double* a, size_t la, const double* b, size_t lb, int c, uint32_t r, std::vector<double>* D) {
    D->assign(la * lb, kInf);
    const int64_t A = (int64_t)lb - 1, B = (int64_t)la - 1;
    // (a radius beyond max(la, lb) is the whole matrix; the cap keeps the products inside 64 bits)
    const int64_t w = (int64_t)std::min<uint64_t>(r, std::max(la, lb)) * std::max(A, B);
    for (size_t i = 0; i < la; i++) {
        for (size_t j = 0; j < lb; j++) {
            const int64_t x = (int64_t)i * A - (int64_t)j * B;
            if (r != 0 && (x > w || x < -w)) continue;  // outside the band: +inf
            double cost = 0.0;
            for (int k = 0; k < c; k++) {
                const double d = a[i * c + k] - b[j * c + k];
                cost = cost + d * d;
            }
            double m;
            if (i == 0 && j == 0) m = 0.0;
            else if (i == 0) m = (*D)[j - 1];
            else if (j == 0) m = (*D)[(i - 1) * lb];
            else m = std::fmin(std::fmin((*D)[(i - 1) * lb + j], (*D)[i * lb + j - 1]), (*D)[(i - 1) * lb + j - 1]);
            (*D)[i * lb + j] = cost + m;
        }
    }
}

}  // namespace

extern "C" {

double ref_dtw_band(const double* a, size_t la, const double* b, size_t lb, int c, uint32_t r) {
    if (la == 0 || lb == 0) return kInf;
    static thread_local std::vector<double> D;
    band_matrix(a, la, b, lb, c, r, &D);
    return D[la * lb - 1] / (double)(la + lb);
}

// 1 iff (i, j) lies inside the band of radius r >= 1 of a pair of lengths (la, lb)
int ref_in_band(size_t i, size_t j, size_t la, size_t lb, uint32_t r) {
    const int64_t A = (int64_t)lb - 1, B = (int64_t)la - 1;
    const int64_t w = (int64_t)std::min<uint64_t>(r, std::max(la, lb)) * std::max(A, B);
    const int64_t x = (int64_t)i * A - (int64_t)j * B;
    return x <= w && x >= -w;
}

// orc_dtw_topk with the banded distance: frame offsets (nseg + 1 entries, in FRAMES); for each query the k smallest
// (distance, index), ascending; NaN / inf never win; unfilled slots = (inf, 0xFFFFFFFF). Queries are spread over threads.
void ref_dtw_band_topk(const double* dict, const uint64_t* dict_off, size_t nseg, const double* q, const uint64_t* q_off, size_t nq, int c,
                       int k, uint32_t r, int nthreads, uint32_t* out_idx, double* out_dist) {
    auto one = [&](size_t qi) {
        std::vector<std::pair<double, uint32_t>> best;
        const double* qa = q + q_off[qi] * c;
        const size_t lq = (size_t)(q_off[qi + 1] - q_off[qi]);
        for (size_t d = 0; d < nseg; d++) {
            const double dist = ref_dtw_band(qa, lq, dict + dict_off[d] * c, (size_t)(dict_off[d + 1] - dict_off[d]), c, r);
            if (!(dist < kInf)) continue;
            std::pair<double, uint32_t> cand(dist, (uint32_t)d);
            if ((int)best.size() < k) {
                best.insert(std::upper_bound(best.begin(), best.end(), cand), cand);
            } else if (cand < best.back()) {
                best.pop_back();
                best.insert(std::upper_bound(best.begin(), best.end(), cand), cand);
            }
        }
        for (int s = 0; s < k; s++) {
            out_idx[qi * k + s] = s < (int)best.size() ? best[s].second : 0xFFFFFFFFu;
            out_dist[qi * k + s] = s < (int)best.size() ? best[s].first : kInf;
        }
    };
    std::vector<std::thread> th;
    for (int t = 0; t < std::max(nthreads, 1); t++)
        th.emplace_back([&, t] {
            for (size_t qi = t; qi < nq; qi += std::max(nthreads, 1)) one(qi);
        });
    for (auto& x : th) x.join();
}

// the banded warping path: (i, j) pairs in ascending order (capacity la + lb - 1 pairs); returns its length, 0 if a side is
// empty or the distance is not finite. The backtrack is tests/cpp/dtw_path.cpp's.
size_t ref_dtw_band_path(const double* a, size_t la, const double* b, size_t lb, int c, uint32_t r, uint32_t* out_ij) {
    if (la == 0 || lb == 0) return 0;
    std::vector<double> D;
    band_matrix(a, la, b, lb, c, r, &D);
    if (!std::isfinite(D[la * lb - 1] / (double)(la + lb))) return 0;
    std::vector<uint32_t> rev;
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
            const double m = std::fmin(std::fmin(up, left), diag);
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
