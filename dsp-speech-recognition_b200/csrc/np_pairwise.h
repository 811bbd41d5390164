// NumPy's pairwise summation of float64 (pairwise_sum in numpy/_core/src/umath/loops_utils.h.src), the order in which
// np.sum / np.mean add a contiguous 1-D array.  One rule for every caller: the helper kernels (helpers.cu np_sum_any),
// the float-sample endpoint statistics (endpoint_kernel.cuh K2f) and the exact autocorrelation of float frames (acr_lag,
// K3r's float gate) take their leaves, splits, block sums and tree walk from here.
//   n <= kNpPairwiseBlock  one leaf: pairwise_block;
//   n >  kNpPairwiseBlock  sum(first n2) + sum(rest) with n2 = np_pairwise_split(n), recursively (pairwise_walk).
#pragma once

#ifdef __CUDACC__
#define NP_HD __host__ __device__ inline
#else
#define NP_HD inline
#endif

namespace dspfe {

constexpr int kNpPairwiseBlock = 128;   // PW_BLOCKSIZE

// where a run longer than kNpPairwiseBlock is split: n / 2 rounded down to a multiple of 8
NP_HD int np_pairwise_split(int n) {
    int n2 = n / 2;
    n2 -= n2 % 8;
    return n2;
}

// one leaf (n <= kNpPairwiseBlock): term(i) is the i-th addend.  Below 8 terms a plain loop; otherwise eight interleaved
// accumulators over the first n - n % 8 terms, ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the remainder in order.
template <class F>
NP_HD double pairwise_block(F term, int n) {
    if (n < 8) { double r = 0.; for (int i = 0; i < n; ++i) r += term(i); return r; }
    double r0 = term(0), r1 = term(1), r2 = term(2), r3 = term(3), r4 = term(4), r5 = term(5), r6 = term(6), r7 = term(7);
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
        r0 += term(i); r1 += term(i + 1); r2 += term(i + 2); r3 += term(i + 3);
        r4 += term(i + 4); r5 += term(i + 5); r6 += term(i + 6); r7 += term(i + 7);
    }
    double res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
    for (; i < n; ++i) res += term(i);
    return res;
}

// any n: the split tree walked in post order without recursion (explicit stack of pending right halves; the device stack
// stays small).  p0 is the position of the first term (a pointer or an index: it only needs p + k), leaf(p, m) sums the m <=
// kNpPairwiseBlock terms from position p.  24 levels cover every int n.
template <class Pos, class Leaf>
NP_HD double pairwise_walk(Pos p0, int n, Leaf leaf) {
    struct Item { Pos p; int n; int state; double left; };
    Item st[24];
    int sp = 0;
    st[0] = {p0, n, 0, 0.};
    double ret = 0.;
    while (sp >= 0) {
        Item& t = st[sp];
        if (t.n <= kNpPairwiseBlock) { ret = leaf(t.p, t.n); --sp; continue; }
        const int n2 = np_pairwise_split(t.n);
        if (t.state == 0) { t.state = 1; st[++sp] = {t.p, n2, 0, 0.}; }
        else if (t.state == 1) { t.left = ret; t.state = 2; st[++sp] = {t.p + n2, t.n - n2, 0, 0.}; }
        else { ret = t.left + ret; --sp; }
    }
    return ret;
}

// np.sum of term(0) .. term(n - 1) for any n
template <class F>
NP_HD double np_pairwise_sum_any(F term, int n) {
    return pairwise_walk(0, n, [term](int p, int m) { return pairwise_block([term, p](int i) { return term(p + i); }, m); });
}

}  // namespace dspfe
