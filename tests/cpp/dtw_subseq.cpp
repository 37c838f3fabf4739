// Subsequence DTW: the checker of ss_dict_locate (tests/test_locate_*.py). CPU, f64, built by tests/subseq_reference.py with
// -ffp-contract=off like the oracle, so that mul and add stay separate IEEE operations.
//
// Spec (A12, DESIGN.md §3.1g; extends oracle/ASSUMPTIONS.h A8). For a query a of La frames and a segment b of Lb frames, c(i, j) is
// A8's local cost and
//     S(0, j) = c(0, j) + 0.0                                   (the path may start at any column)
//     S(i, j) = c(i, j) + fmin(fmin(S(i-1, j), S(i, j-1)), S(i-1, j-1))      i >= 1, a missing neighbour (j = 0) +inf
// st(0, j) = j; st(i, j) = st of the neighbour align_dir's rule picks (diag if it equals the min, else up if it does, else left).
// The end e is the smallest j whose S(La-1, j) is the minimum of the finite values of row La-1; the hit is (S(La-1, e),
// st(La-1, e), e). No finite value, La = 0 or Lb = 0: no hit. The top-k ranks the hits of a query by (cost, index).
//
// S is computed with the operations of orc_dtw (oracle/soundsym_oracle.cpp) in the same order: the cost accumulated coefficient by
// coefficient, cost + m. ref_dtw_matrix is A8's D itself (orc_dtw's matrix, unnormalised), for the identities of DESIGN.md §3.1g.
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
constexpr uint32_t kNone = 0xFFFFFFFFu;

double local_cost(const double* a, size_t i, const double* b, size_t j, int c) {
    double cost = 0.0;
    for (int k = 0; k < c; k++) {
        const double d = a[i * c + k] - b[j * c + k];
        cost = cost + d * d;
    }
    return cost;
}

// S and st (la x lb, la, lb >= 1)
void subseq_matrix(const double* a, size_t la, const double* b, size_t lb, int c, std::vector<double>* S, std::vector<uint32_t>* st) {
    S->assign(la * lb, kInf);
    st->assign(la * lb, kNone);
    for (size_t i = 0; i < la; i++) {
        for (size_t j = 0; j < lb; j++) {
            const double cost = local_cost(a, i, b, j, c);
            double m;
            uint32_t s;
            if (i == 0) {
                m = 0.0;
                s = (uint32_t)j;
            } else {
                const double up = (*S)[(i - 1) * lb + j];
                const double left = j ? (*S)[i * lb + j - 1] : kInf;
                const double diag = j ? (*S)[(i - 1) * lb + j - 1] : kInf;
                m = std::fmin(std::fmin(up, left), diag);
                if (diag == m) s = (*st)[(i - 1) * lb + j - 1];
                else if (up == m) s = (*st)[(i - 1) * lb + j];
                else s = j ? (*st)[i * lb + j - 1] : kNone;
            }
            (*S)[i * lb + j] = cost + m;
            (*st)[i * lb + j] = s;
        }
    }
}

// the hit of row la - 1; false if it has no finite value
bool subseq_hit(const std::vector<double>& S, const std::vector<uint32_t>& st, size_t la, size_t lb, double* cost, uint32_t* start, uint32_t* end) {
    *cost = kInf, *start = kNone, *end = kNone;
    for (size_t j = 0; j < lb; j++) {
        const double v = S[(la - 1) * lb + j];
        if (v < *cost) *cost = v, *end = (uint32_t)j, *start = st[(la - 1) * lb + j];
    }
    return *end != kNone;
}

}  // namespace

extern "C" {

// the hit of one pair: returns 1 and (cost, start, end), or 0 and (inf, 0xFFFFFFFF, 0xFFFFFFFF). out_S / out_st (la x lb) may be NULL.
int ref_subseq(const double* a, size_t la, const double* b, size_t lb, int c, double* out_S, uint32_t* out_st, double* cost, uint32_t* start,
               uint32_t* end) {
    *cost = kInf, *start = kNone, *end = kNone;
    if (la == 0 || lb == 0) return 0;
    std::vector<double> S;
    std::vector<uint32_t> st;
    subseq_matrix(a, la, b, lb, c, &S, &st);
    if (out_S) std::copy(S.begin(), S.end(), out_S);
    if (out_st) std::copy(st.begin(), st.end(), out_st);
    return subseq_hit(S, st, la, lb, cost, start, end) ? 1 : 0;
}

// A8's unnormalised D (la x lb, la, lb >= 1), orc_dtw's operations in orc_dtw's order
void ref_dtw_matrix(const double* a, size_t la, const double* b, size_t lb, int c, double* out_D) {
    for (size_t i = 0; i < la; i++)
        for (size_t j = 0; j < lb; j++) {
            const double cost = local_cost(a, i, b, j, c);
            double m;
            if (i == 0 && j == 0) m = 0.0;
            else if (i == 0) m = out_D[j - 1];
            else if (j == 0) m = out_D[(i - 1) * lb];
            else m = std::fmin(std::fmin(out_D[(i - 1) * lb + j], out_D[i * lb + j - 1]), out_D[(i - 1) * lb + j - 1]);
            out_D[i * lb + j] = cost + m;
        }
}

// the backtrack of S from the hit's end (la - 1, e) to row 0 under align_dir's rule: (i, j) pairs in ascending order, j a
// column of the segment (capacity la + lb - 1 pairs); returns its length, 0 if the pair has no hit
size_t ref_subseq_path(const double* a, size_t la, const double* b, size_t lb, int c, uint32_t* out_ij) {
    if (la == 0 || lb == 0) return 0;
    std::vector<double> S;
    std::vector<uint32_t> st;
    subseq_matrix(a, la, b, lb, c, &S, &st);
    double cost;
    uint32_t start, end;
    if (!subseq_hit(S, st, la, lb, &cost, &start, &end)) return 0;
    std::vector<uint32_t> rev;
    size_t i = la - 1, j = end;
    for (;;) {
        rev.push_back((uint32_t)i);
        rev.push_back((uint32_t)j);
        if (i == 0) break;
        const double up = S[(i - 1) * lb + j];
        const double left = j ? S[i * lb + j - 1] : kInf;
        const double diag = j ? S[(i - 1) * lb + j - 1] : kInf;
        const double m = std::fmin(std::fmin(up, left), diag);
        if (diag == m) i--, j--;
        else if (up == m) i--;
        else j--;
    }
    const size_t n = rev.size() / 2;
    for (size_t s = 0; s < n; s++) {
        out_ij[2 * s] = rev[2 * (n - 1 - s)];
        out_ij[2 * s + 1] = rev[2 * (n - 1 - s) + 1];
    }
    return n;
}

// every query against every segment (frame offsets, nseg + 1 entries): the k best hits by (cost, index), ascending; unfilled
// slots (0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, inf). Local indices. Queries are spread over threads.
void ref_subseq_topk(const double* dict, const uint64_t* dict_off, size_t nseg, const double* q, const uint64_t* q_off, size_t nq, int c, int k,
                     int nthreads, uint32_t* out_idx, uint32_t* out_start, uint32_t* out_end, double* out_cost) {
    auto one = [&](size_t qi) {
        std::vector<std::pair<double, uint32_t>> best;
        std::vector<std::pair<uint32_t, uint32_t>> spans(nseg);
        const double* qa = q + q_off[qi] * c;
        const size_t lq = (size_t)(q_off[qi + 1] - q_off[qi]);
        for (size_t d = 0; d < nseg; d++) {
            double cost;
            uint32_t s, e;
            if (!ref_subseq(qa, lq, dict + dict_off[d] * c, (size_t)(dict_off[d + 1] - dict_off[d]), c, nullptr, nullptr, &cost, &s, &e)) continue;
            spans[d] = {s, e};
            std::pair<double, uint32_t> cand(cost, (uint32_t)d);
            if ((int)best.size() < k) {
                best.insert(std::upper_bound(best.begin(), best.end(), cand), cand);
            } else if (cand < best.back()) {
                best.pop_back();
                best.insert(std::upper_bound(best.begin(), best.end(), cand), cand);
            }
        }
        for (int s = 0; s < k; s++) {
            const bool f = s < (int)best.size();
            out_idx[qi * k + s] = f ? best[s].second : kNone;
            out_start[qi * k + s] = f ? spans[best[s].second].first : kNone;
            out_end[qi * k + s] = f ? spans[best[s].second].second : kNone;
            out_cost[qi * k + s] = f ? best[s].first : kInf;
        }
    };
    std::vector<std::thread> th;
    for (int t = 0; t < std::max(nthreads, 1); t++)
        th.emplace_back([&, t] {
            for (size_t qi = t; qi < nq; qi += std::max(nthreads, 1)) one(qi);
        });
    for (auto& x : th) x.join();
}

}  // extern "C"
