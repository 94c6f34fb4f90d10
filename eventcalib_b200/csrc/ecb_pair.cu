// k_pair — candidate circles of one window from the kept clusters of both polarities
// (CirclesEventFrame::extractFeatures, CirclesEventFrame.cpp:137-312) and the batched Kasa circle fit
// (CirclesEventFrame::fitCircle, CirclesEventFrame.cpp:361-415).  One CTA per window at a time.  Small windows (member
// pixels staged in shared memory, <= PAIR_LANE_MAX_POINTS points per polarity) run one LANE per positive cluster in
// 64-thread CTAs: each lane does its cluster's k-NN over the medians (one pass keeping the k smallest keys), Kasa fits and
// fit errors (one sequential sum, like the reference's fitErr) alone.  Larger windows and kept-cluster tables in global
// scratch run one WARP per positive cluster in 256-thread CTAs: k-NN by warp arg-min, fit errors summed warp-wide.  The
// k-NN replaces the nanoflann trees (:160-168); ties -> lowest index.
//
// This translation unit is compiled with -fmad=false: the reference is built without FMA contraction
// (CMakeLists.txt:6-19, x86-64 baseline), and the 3x3 LU / fit-error arithmetic below follows it operation
// by operation.  The 9 moment sums are exact integers (int64 in k_cluster), so A and b are bit-identical.
#include <float.h>

#include <algorithm>

#include "ecb_window.cuh"

namespace {

constexpr int PAIR_THREADS = 256;
constexpr int KNN_MAX = 8;
#ifndef ECB_PAIR_KM
#define ECB_PAIR_KM 3      // capacity of the candidate arrays of the small variant (the reference's knn_num)
#endif
#ifndef ECB_PAIR_JROLL
#define ECB_PAIR_JROLL 1   // the per-candidate loop of the pair evaluation stays rolled (63 -> 47 KB of SASS, 0.98 -> 0.91 ms)
#endif
#ifndef ECB_PAIR_KM4
#define ECB_PAIR_KM4 1  // knn_num <= ECB_PAIR_KM: small candidate arrays, a fraction of the unrolled code
#endif
// lane per cluster: 64-thread CTAs (~40 positive clusters per DAVIS346 window), 8 of them resident per SM (<= 128 registers)
constexpr int PAIR_LANE_THREADS = 64, PAIR_LANE_CTAS = 8;
// one lane sums a cluster's members alone: that pays while clusters are a few dozen members wide (DAVIS346 1.5 ms windows,
// ~1 200 points and ~30-member clusters per polarity).  Larger problems (VGA 10 ms windows: ~8 800 points, ~180-member
// clusters) keep a warp per cluster
constexpr int PAIR_LANE_MAX_POINTS = 4096;

// Eigen PartialPivLU<Matrix3d>::solve, unblocked, first-max pivot [external: Eigen, not in /root/reference]
// (kept out of line, like warp_abs_dev / warp_knn: k_pair inlined was 180 KB of SASS and stalled on instruction fetch)
__device__ __noinline__ void lu_solve3(double A[3][3], const double b_in[3], double x[3]) {
    int perm[3] = {0, 1, 2};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        int piv = k;
        double big = fabs(A[k][k]);
        for (int i = k + 1; i < 3; ++i)
            if (fabs(A[i][k]) > big) {
                big = fabs(A[i][k]);
                piv = i;
            }
        if (big != 0.0) {
            if (piv != k) {
                for (int j = 0; j < 3; ++j) {
                    double t = A[k][j];
                    A[k][j] = A[piv][j];
                    A[piv][j] = t;
                }
                int t = perm[k];
                perm[k] = perm[piv];
                perm[piv] = t;
            }
            for (int i = k + 1; i < 3; ++i) A[i][k] /= A[k][k];
        }
        for (int i = k + 1; i < 3; ++i)
            for (int j = k + 1; j < 3; ++j) A[i][j] -= A[i][k] * A[k][j];
    }
    double y[3] = {b_in[perm[0]], b_in[perm[1]], b_in[perm[2]]};
    y[1] -= A[1][0] * y[0];
    y[2] -= (A[2][0] * y[0] + A[2][1] * y[1]);
    y[2] /= A[2][2];
    y[1] -= A[1][2] * y[2];
    y[1] /= A[1][1];
    y[0] -= (A[0][1] * y[1] + A[0][2] * y[2]);
    y[0] /= A[0][0];
    x[0] = y[0];
    x[1] = y[1];
    x[2] = y[2];
}

// m = Sx Sy Sxx Syy Sxy Sxxx Syyy Sxyy Sxxy, N = sample count   (CirclesEventFrame.cpp:406-414)
__device__ void fit_from_moments(const double *m, double N, double &cx, double &cy, double &r) {
    double A[3][3] = {{2 * m[0], 2 * m[1], N}, {2 * m[2], 2 * m[4], m[0]}, {2 * m[4], 2 * m[3], m[1]}};
    double b[3] = {m[2] + m[3], m[5] + m[7], m[8] + m[6]};
    double x[3];
    lu_solve3(A, b, x);
    cx = x[0];
    cy = x[1];
    r = sqrt(x[0] * x[0] + x[1] * x[1] + x[2]);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// sum over the members of |‖p-c‖ - r|   (CirclesEventFrame.cpp:209-214,300-305)
// DIRECT: `mem` already holds the members' packed pixels (staged in shared memory); else it holds pids into `pts`
template <bool DIRECT>
__device__ __noinline__ double warp_abs_dev(const uint32_t *pts, const uint32_t *mem, int sz, double cx, double cy, double r) {
    double s = 0;
#pragma unroll 1  // clusters rarely exceed one warp's width; the unrolled FP64 sqrt bodies only cost instruction cache
    for (int i = threadIdx.x & 31; i < sz; i += 32) {
        const uint32_t p = DIRECT ? mem[i] : pts[mem[i]];
        const double dx = (double) ECB_PIX_X(p) - cx, dy = (double) ECB_PIX_Y(p) - cy;
        s += fabs(sqrt(dx * dx + dy * dy) - r);
    }
    return warp_sum(s);
}

// sum over the members of |‖p-c‖ - r|, positive members then negative members into one accumulator, then one division
// (CirclesEventFrame.cpp:209-214,300-305): one lane, one member at a time, over the staged pixels in member-list order
__device__ __noinline__ double lane_fit_err(const uint32_t *pixP, int szP, const uint32_t *pixN, int szN, double cx, double cy,
                                            double r) {
    double e = 0;
    const int tot = szP + szN;
#pragma unroll 1  // unrolled by 4 it needs more than the 128 registers of 8 resident CTAs (0.60 -> 0.58 ms at 7 CTAs)
    for (int i = 0; i < tot; ++i) {
        const uint32_t p = i < szP ? pixP[i] : pixN[i - szP];
        const double dx = (double) ECB_PIX_X(p) - cx, dy = (double) ECB_PIX_Y(p) - cy;
        e += fabs(sqrt(dx * dx + dy * dy) - r);
    }
    return e / ((double) tot * r);
}

// the KM nearest medians of (qx, qy) for one lane, in one pass: keys (squared distance << 32 | index), ascending; unused
// slots stay ~0.  Every lane walks the same table in the same order, so the median reads are broadcasts.
template <int KM>
__device__ __forceinline__ void lane_knn(const int *mx, const int *my, int n, int qx, int qy, unsigned long long (&key)[KM]) {
#pragma unroll
    for (int q = 0; q < KM; ++q) key[q] = ~0ull;
#pragma unroll 1
    for (int i = 0; i < n; ++i) {
        const long long dx = qx - mx[i], dy = qy - my[i];
        const unsigned long long k = ((unsigned long long) (dx * dx + dy * dy) << 32) | (unsigned) i;
        if (k < key[KM - 1]) {  // keys are unique (they carry the index): ties go to the lower index
#pragma unroll
            for (int q = KM - 1; q > 0; --q) key[q] = k < key[q - 1] ? key[q - 1] : (k < key[q] ? k : key[q]);
            key[0] = k < key[0] ? k : key[0];
        }
    }
}

template <int KM>
__device__ __forceinline__ unsigned long long pick(const unsigned long long (&key)[KM], int j) {
    unsigned long long v = key[0];
#pragma unroll
    for (int q = 1; q < KM; ++q)
        if (j == q) v = key[q];
    return v;
}

// the reference's `real` cut over the first K neighbours: the first one farther than 4x the nearest or than the gate
template <int KM>
__device__ __forceinline__ int knn_real(const unsigned long long (&key)[KM], int K, double gate) {
    int real = K;
    const double d0 = (double) (key[0] >> 32);
#pragma unroll
    for (int q = KM - 1; q >= 0; --q) {
        const double d = (double) (key[q] >> 32);
        if (q < K && (d > d0 * 4 || d > gate)) real = q;
    }
    return real;
}

// k nearest medians (ascending squared distance, ties by index), warp cooperative
__device__ __noinline__ void warp_knn(const int *mx, const int *my, int n, int qx, int qy, int k, int *idx, unsigned long long *d2) {
    // key = (squared distance, index); the k smallest keys in ascending order.  n <= 64 (the usual case: ~40 kept clusters):
    // every lane computes its two keys once, each round is one warp min over registers
    const int lane = threadIdx.x & 31;
    unsigned long long last = 0;
    bool first = true;
    if (n <= 64) {
        unsigned long long key0 = ~0ull, key1 = ~0ull;
        if (lane < n) {
            const long long dx = qx - mx[lane], dy = qy - my[lane];
            key0 = ((unsigned long long) (dx * dx + dy * dy) << 32) | (unsigned) lane;
        }
        if (lane + 32 < n) {
            const long long dx = qx - mx[lane + 32], dy = qy - my[lane + 32];
            key1 = ((unsigned long long) (dx * dx + dy * dy) << 32) | (unsigned) (lane + 32);
        }
        for (int j = 0; j < k; ++j) {
            unsigned long long best = key0 < key1 ? key0 : key1;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long t = __shfl_xor_sync(0xffffffffu, best, o);
                best = t < best ? t : best;
            }
            idx[j] = best == ~0ull ? -1 : (int) (best & 0xFFFFFFFFu);
            d2[j] = best >> 32;
            if (key0 == best) key0 = ~0ull;  // keys are unique (they carry the index)
            if (key1 == best) key1 = ~0ull;
        }
        return;
    }
    for (int j = 0; j < k; ++j) {
        unsigned long long best = ~0ull;
#pragma unroll 1
        for (int i = lane; i < n; i += 32) {
            const long long dx = qx - mx[i], dy = qy - my[i];
            const unsigned long long key = ((unsigned long long) (dx * dx + dy * dy) << 32) | (unsigned) i;
            if ((first || key > last) && key < best) best = key;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            unsigned long long t = __shfl_xor_sync(0xffffffffu, best, o);
            best = t < best ? t : best;
        }
        idx[j] = best == ~0ull ? -1 : (int) (best & 0xFFFFFFFFu);
        d2[j] = best >> 32;
        last = best;
        first = false;
    }
}

// Per-CTA tables over the kept clusters (max_k entries each): accepted circle (3 doubles), medians of both polarities,
// accepted negative partner.  GT = false: in dynamic shared memory (pointers derived from the shared array only);
// GT = true (very many kept clusters, e.g. noisy 1280x720 windows): in per-CTA global scratch.
// KM: capacity of the per-warp candidate arrays (>= knn_num).  The kernel is instruction-cache bound (ncu: 110 KB of SASS,
// `no_instruction` the second largest stall at 4.8 per issue): the reference's default is 3 neighbours, and KM = 3 instead of 8
// together with the un-unrolled member / staging / candidate loops takes the code to 47 KB and the kernel from 1.25 to 0.91 ms
// (profiles/r2t_pair_code_size.md; folding the two candidate passes into one loop body — 50 KB — was slower again: 1.04 ms)
template <bool DIRECT, bool FIT, bool GT, int KM, bool LANE>
__global__ void __launch_bounds__(LANE ? PAIR_LANE_THREADS : PAIR_THREADS, LANE ? PAIR_LANE_CTAS : 4) k_pair(const PairArgs a) {
    constexpr int NT = LANE ? PAIR_LANE_THREADS : PAIR_THREADS;
    static_assert(!LANE || (DIRECT && !GT), "lane per cluster reads the staged member pixels");
    extern __shared__ __align__(16) uint32_t sm_dyn[];
    double (*acc_c)[3];
    if constexpr (GT) acc_c = reinterpret_cast<double (*)[3]>(a.gtab + (size_t) blockIdx.x * a.gtab_stride);
    else acc_c = reinterpret_cast<double (*)[3]>(sm_dyn);
    int *const tab_i = reinterpret_cast<int *>(acc_c + a.max_k);
    int *const mx[2] = {tab_i, tab_i + a.max_k}, *const my[2] = {tab_i + 2 * a.max_k, tab_i + 3 * a.max_k};
    int *const acc_ni = tab_i + 4 * a.max_k;
    uint32_t *const sm_pix = GT ? sm_dyn : reinterpret_cast<uint32_t *>(acc_ni + a.max_k);  // DIRECT: member pixels of both polarities
    __shared__ uint32_t ws[33];
    __shared__ int s_next;  // next unclaimed positive cluster of the window (the clusters' fit work varies: dynamic hand-out)
    const int tid = threadIdx.x, lane = tid & 31;

    __shared__ int s_win;
    for (int w = blockIdx.x;; w += gridDim.x) {
        if (a.win_counter) {  // dynamic hand-out: the windows' pairing work varies by a factor of two
            __syncthreads();
            if (tid == 0) s_win = (int) atomicAdd(a.win_counter, 1u);
            __syncthreads();
            w = s_win;
        }
        if (w >= a.n_win) break;
        const ProbDesc dn = a.prob[2 * w], dp = a.prob[2 * w + 1];
        const ProbHdr hn = a.hdr[2 * w], hp = a.hdr[2 * w + 1];
        const KeptCluster *kn = a.ktab + (size_t) (2 * w) * a.max_k, *kp = a.ktab + (size_t) (2 * w + 1) * a.max_k;
        const int nkn = hn.n_kept, nkp = hp.n_kept;
        __syncthreads();
#pragma unroll 1
        for (int i = tid; i < nkn; i += NT) {
            mx[0][i] = kn[i].med_x;
            my[0][i] = kn[i].med_y;
        }
#pragma unroll 1
        for (int i = tid; i < nkp; i += NT) {
            mx[1][i] = kp[i].med_x;
            my[1][i] = kp[i].med_y;
            acc_ni[i] = -1;
        }
        if (tid == 0) s_next = 0;
        __syncthreads();
        const bool enough0 = dn.n > 0 && dp.n > 0 && (uint32_t) nkp >= a.rows_cols && (uint32_t) nkn >= a.rows_cols;
        const bool enough = enough0;
        const uint32_t *ptsP = a.pts[1] + dp.off, *ptsN = a.pts[0] + dn.off;
        const uint32_t *memP = a.kmem[1] + dp.off, *memN = a.kmem[0] + dn.off;
        if (DIRECT && enough0) {
            // stage the kept clusters' member pixels once (coalesced list read, gathered pixel read), then every
            // fit-error loop runs out of shared memory
            const int totP = nkp ? kp[nkp - 1].mem_off + kp[nkp - 1].size : 0, totN = nkn ? kn[nkn - 1].mem_off + kn[nkn - 1].size : 0;
#pragma unroll LANE ? 4 : 1  // a small CTA needs several gathers in flight per thread
            for (int i = tid; i < totN; i += NT) sm_pix[i] = ptsN[memN[i]];
#pragma unroll LANE ? 4 : 1
            for (int i = tid; i < totP; i += NT) sm_pix[a.smem_cap + i] = ptsP[memP[i]];
            memN = sm_pix;
            memP = sm_pix + a.smem_cap;
            __syncthreads();
        }
        const double gate = 4 * a.rthr * a.rthr;
        if (LANE && enough) {
            // one lane carries one positive cluster through the whole pipeline: acc_ni[pi] depends on pi alone
#pragma unroll 1
            for (int pi = tid; pi < nkp; pi += NT) {
                if (!FIT) {  // CirclesEventFrame.cpp:282-312
                    unsigned long long key[1];
                    lane_knn<1>(mx[0], my[0], nkn, mx[1][pi], my[1][pi], key);
                    if ((double) (key[0] >> 32) > gate) continue;
                    const int n0 = (int) (unsigned) key[0];
                    lane_knn<1>(mx[1], my[1], nkp, mx[0][n0], my[0][n0], key);
                    if ((int) (unsigned) key[0] != pi) continue;
                    const double px = mx[1][pi], py = my[1][pi], qx = mx[0][n0], qy = my[0][n0];
                    const double cx = (px + qx) / 2, cy = (py + qy) / 2;
                    const double ddx = px - qx, ddy = py - qy;
                    const double r = sqrt(ddx * ddx + ddy * ddy) / 2;
                    const double e = lane_fit_err(memP + kp[pi].mem_off, kp[pi].size, memN + kn[n0].mem_off, kn[n0].size, cx, cy, r);
                    if (e < 10 / r) {
                        acc_ni[pi] = n0;
                        acc_c[pi][0] = cx;
                        acc_c[pi][1] = cy;
                        acc_c[pi][2] = r;
                    }
                } else {  // CirclesEventFrame.cpp:180-281
                    const int K = min(min(a.knn_num, KM), min(nkn, nkp));
                    // the best of the first `real` candidate pairs, (pi, key[j]) or (key[j], nsel), as the reference's
                    // min_element over fitErrs; the (pi, nsel) fit of the first pass is memoised like the reference's fit
                    // cache (CirclesEventFrame.cpp:199-225)
                    double b_err = 0, b_cx = 0, b_cy = 0, b_r = 0, m_err = 0, m_cx = 0, m_cy = 0, m_r = 0;
                    int b_c = 0;
                    auto best_pair = [&](const unsigned long long (&key)[KM], int real, bool rev, int fixed) {
#pragma unroll 1
                        for (int j = 0; j < real; ++j) {
                            const int c = (int) (unsigned) pick(key, j);
                            const int p = rev ? c : fixed, n = rev ? fixed : c;
                            double e, cx, cy, r;
                            if (rev && p == pi) {  // same pair, same numbers
                                e = m_err, cx = m_cx, cy = m_cy, r = m_r;
                            } else {
                                double m[9];
#pragma unroll
                                for (int q = 0; q < 9; ++q) m[q] = kp[p].m[q] + kn[n].m[q];
                                fit_from_moments(m, (double) (kp[p].size + kn[n].size), cx, cy, r);
                                const double ddx = (double) mx[1][p] - (double) mx[0][n], ddy = (double) my[1][p] - (double) my[0][n];
                                const double approx = sqrt(ddx * ddx + ddy * ddy) / 2;
                                e = r > a.rthr || r > 2 * approx
                                        ? DBL_MAX
                                        : lane_fit_err(memP + kp[p].mem_off, kp[p].size, memN + kn[n].mem_off, kn[n].size, cx, cy, r);
                            }
                            if (j == 0 || e < b_err) b_err = e, b_cx = cx, b_cy = cy, b_r = r, b_c = c;
                        }
                    };
                    unsigned long long key[KM];
                    lane_knn<KM>(mx[0], my[0], nkn, mx[1][pi], my[1][pi], key);
                    int real = knn_real(key, K, gate);
                    if (real == 0) continue;
                    best_pair(key, real, false, pi);
                    if (!(b_err < 2 / b_r)) continue;
                    const int nsel = b_c;
                    m_err = b_err, m_cx = b_cx, m_cy = b_cy, m_r = b_r;
                    lane_knn<KM>(mx[1], my[1], nkp, mx[0][nsel], my[0][nsel], key);
                    real = knn_real(key, K, gate);
                    if (real == 0) continue;
                    best_pair(key, real, true, nsel);
                    if (b_c == pi) {
                        acc_ni[pi] = nsel;
                        acc_c[pi][0] = b_cx;
                        acc_c[pi][1] = b_cy;
                        acc_c[pi][2] = b_r;
                    }
                }
            }
        } else if (!LANE && enough) {
            for (;;) {
                int pi = 0;
                if (lane == 0) pi = atomicAdd(&s_next, 1);
                pi = __shfl_sync(0xffffffffu, pi, 0);
                if (pi >= nkp) break;
                int nidx[KM], pidx[KM];
                unsigned long long d2[KM];
                if (!FIT) {  // CirclesEventFrame.cpp:282-312
                    warp_knn(mx[0], my[0], nkn, mx[1][pi], my[1][pi], 1, nidx, d2);
                    if ((double) d2[0] > gate) continue;
                    const int n0 = nidx[0];
                    warp_knn(mx[1], my[1], nkp, mx[0][n0], my[0][n0], 1, pidx, d2);
                    if (pidx[0] != pi) continue;
                    const double px = mx[1][pi], py = my[1][pi], qx = mx[0][n0], qy = my[0][n0];
                    const double cx = (px + qx) / 2, cy = (py + qy) / 2;
                    const double ddx = px - qx, ddy = py - qy;
                    const double r = sqrt(ddx * ddx + ddy * ddy) / 2;
                    double e = warp_abs_dev<DIRECT>(ptsP, memP + kp[pi].mem_off, kp[pi].size, cx, cy, r);
                    // the reference accumulates + members then - members into one sum
                    e += warp_abs_dev<DIRECT>(ptsN, memN + kn[n0].mem_off, kn[n0].size, cx, cy, r);
                    e /= (double) (kp[pi].size + kn[n0].size) * r;
                    if (e < 10 / r && lane == 0) {
                        acc_ni[pi] = n0;
                        acc_c[pi][0] = cx;
                        acc_c[pi][1] = cy;
                        acc_c[pi][2] = r;
                    }
                } else {  // CirclesEventFrame.cpp:180-281
                    const int K = min(min(a.knn_num, KM), min(nkn, nkp));
                    double ferr[KM], fr[KM], fcx[KM], fcy[KM];
                    warp_knn(mx[0], my[0], nkn, mx[1][pi], my[1][pi], K, nidx, d2);
                    int real = K;
                    for (int oi = 0; oi < K; ++oi)
                        if ((double) d2[oi] > (double) d2[0] * 4 || (double) d2[oi] > gate) {
                            real = oi;
                            break;
                        }
                    if (real == 0) continue;
                    // Kasa fits of up to `cnt` candidate pairs at once: lane j solves pair j (moments + 3x3 LU, one pass for
                    // all candidates instead of one warp-redundant solve per candidate), the results are broadcast and the
                    // fit error of every pair is then summed warp-wide over its members
                    double s_err = 0, s_cx = 0, s_cy = 0, s_r = 0;  // the fit of (pi, nsel), memoised like the reference's fit
                    bool have_memo = false;                         // cache (CirclesEventFrame.cpp:199-225)
                    auto fit_pairs = [&](const int *plist, const int *nlist, bool p_varies, int cnt) {
                        int p = plist[0], n = nlist[0];
#pragma unroll
                        for (int q = 1; q < KM; ++q)
                            if (lane == q) {
                                if (p_varies) p = plist[q]; else n = nlist[q];
                            }
                        double lcx = 0, lcy = 0, lr = 0;
                        bool lok = false;
                        if (lane < cnt) {
                            double m[9];
#pragma unroll
                            for (int q = 0; q < 9; ++q) m[q] = kp[p].m[q] + kn[n].m[q];
                            fit_from_moments(m, (double) (kp[p].size + kn[n].size), lcx, lcy, lr);
                            const double ddx = (double) mx[1][p] - (double) mx[0][n], ddy = (double) my[1][p] - (double) my[0][n];
                            const double approx = sqrt(ddx * ddx + ddy * ddy) / 2;
                            lok = !(lr > a.rthr || lr > 2 * approx);
                        }
#if ECB_PAIR_JROLL
#pragma unroll 1
#endif
                        for (int j = 0; j < cnt; ++j) {
                            const int pj = p_varies ? plist[j] : plist[0], nj = p_varies ? nlist[0] : nlist[j];
                            fcx[j] = __shfl_sync(0xffffffffu, lcx, j);
                            fcy[j] = __shfl_sync(0xffffffffu, lcy, j);
                            fr[j] = __shfl_sync(0xffffffffu, lr, j);
                            const int okj = __shfl_sync(0xffffffffu, (int) lok, j);
                            if (have_memo && pj == pi) {  // same pair, same numbers
                                ferr[j] = s_err;
                                fcx[j] = s_cx;
                                fcy[j] = s_cy;
                                fr[j] = s_r;
                                continue;
                            }
                            if (!okj) {
                                ferr[j] = DBL_MAX;
                                continue;
                            }
                            double e = warp_abs_dev<DIRECT>(ptsP, memP + kp[pj].mem_off, kp[pj].size, fcx[j], fcy[j], fr[j]);
                            e += warp_abs_dev<DIRECT>(ptsN, memN + kn[nj].mem_off, kn[nj].size, fcx[j], fcy[j], fr[j]);
                            ferr[j] = e / ((double) (kp[pj].size + kn[nj].size) * fr[j]);
                        }
                    };
                    fit_pairs(&pi, nidx, false, real);
                    int nmin = 0;
                    for (int j = 1; j < real; ++j)
                        if (ferr[j] < ferr[nmin]) nmin = j;
                    if (!(ferr[nmin] < 2 / fr[nmin])) continue;
                    const int nsel = nidx[nmin];
                    s_err = ferr[nmin], s_cx = fcx[nmin], s_cy = fcy[nmin], s_r = fr[nmin];
                    have_memo = true;
                    warp_knn(mx[1], my[1], nkp, mx[0][nsel], my[0][nsel], K, pidx, d2);
                    real = K;
                    for (int oi = 0; oi < K; ++oi)
                        if ((double) d2[oi] > (double) d2[0] * 4 || (double) d2[oi] > gate) {
                            real = oi;
                            break;
                        }
                    if (real == 0) continue;
                    fit_pairs(pidx, &nsel, true, real);
                    int pmin = 0;
                    for (int i = 1; i < real; ++i)
                        if (ferr[i] < ferr[pmin]) pmin = i;
                    if (pidx[pmin] == pi && lane == 0) {
                        acc_ni[pi] = nsel;
                        acc_c[pi][0] = fcx[pmin];
                        acc_c[pi][1] = fcy[pmin];
                        acc_c[pi][2] = fr[pmin];
                    }
                }
            }
        }
        __syncthreads();
        // ordered compaction (candidates are pushed in ascending pi, CirclesEventFrame.cpp:274-278,306-310)
        uint32_t run = 0;
        double *out = a.cand + (size_t) w * a.cand_stride * 5;
        for (int c0 = 0; c0 < nkp; c0 += NT) {
            const int pi = c0 + tid;
            const bool ok = enough && pi < nkp && acc_ni[pi] >= 0;
            uint32_t tot;
            const uint32_t ex = block_excl_scan(ok ? 1u : 0u, ws, &tot);
            if (ok && run + ex < (uint32_t) a.cand_stride) {
                double *o = out + (size_t) (run + ex) * 5;
                o[0] = pi;
                o[1] = acc_ni[pi];
                o[2] = acc_c[pi][0];
                o[3] = acc_c[pi][1];
                o[4] = acc_c[pi][2];
            }
            run += tot;
        }
        if (tid == 0) {
            ecb_window_summary s;
            s.ev_lo = a.lohi[2 * w];
            s.ev_hi = a.lohi[2 * w + 1] > a.lohi[2 * w] ? a.lohi[2 * w + 1] : a.lohi[2 * w];
            s.n_points[0] = dn.n;
            s.n_points[1] = dp.n;
            s.n_clusters[0] = hn.n_clusters;
            s.n_clusters[1] = hp.n_clusters;
            s.n_kept[0] = nkn;
            s.n_kept[1] = nkp;
            s.n_candidates = (int32_t) run;
            s.status = hn.status | hp.status;
            s.point_offset[0] = dn.off;
            s.point_offset[1] = dp.off;
            a.summary[w] = s;
        }
    }
}

// k_rectify — CirclesEventFrame::rectifyFeatures (CirclesEventFrame.cpp:417-576) for every (kept frame, board circle): one
// warp per circle.  img = the projected centre and four quadrant points of the circle (cv::projectPoints stays with the
// caller, :449): radius search over the window's points (nanoflann radiusSearch: d2 < R2), quadrant-wise +-3 px band
// (:484-519), expansion of the inliers to their whole kept DBSCAN clusters (:522-555; here: a bit mask over the kept-cluster
// table, whose exact integer moments are simply added), Kasa fit (:563-566) and the two sanity gates (:568-574).
struct RectifyArgs {
    const int32_t *win;       // [n_frames] window index of the last front-end run
    int n_frames, n_feat;
    const double *img;        // [n_frames][n_feat][5][2]
    double *out;              // [n_frames][n_feat][3]: cx, cy, r (r < 0: feature deleted)
    const ProbDesc *prob;
    const ProbHdr *hdr;
    const KeptCluster *ktab;
    const uint32_t *pts[2];
    const int32_t *labels[2];
    int max_k;
    double W, H, thr;
};

constexpr int RECT_WARPS = 4;

__global__ void __launch_bounds__(RECT_WARPS * 32) k_rectify(const RectifyArgs a) {
    extern __shared__ uint32_t mask_dyn[];  // [RECT_WARPS][2][mw] bit masks over the kept-cluster tables
    const int mw = (a.max_k + 31) >> 5;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint32_t *const mask[2] = {mask_dyn + (size_t) (2 * wib) * mw, mask_dyn + (size_t) (2 * wib + 1) * mw};
    const int item = blockIdx.x * RECT_WARPS + wib;
    if (item >= a.n_frames * a.n_feat) return;
    const int fr = item / a.n_feat;
    const double *ip = a.img + (size_t) item * 10;
    double *o = a.out + (size_t) item * 3;
    const int w = a.win[fr];
    bool ok = !(ip[0] >= a.W || ip[1] >= a.H || ip[0] < 0 || ip[1] < 0);  // :459-463
    double radius[4], maxRadius = 0;
#pragma unroll
    for (int i = 1; i < 5; ++i) {
        const double dx = ip[2 * i] - ip[0], dy = ip[2 * i + 1] - ip[1];
        radius[i - 1] = sqrt(dx * dx + dy * dy);
        if (radius[i - 1] > maxRadius) maxRadius = radius[i - 1];
    }
    const double R2 = (maxRadius + a.thr) * (maxRadius + a.thr);
    for (int i = lane; i < 2 * mw; i += 32) mask[0][i] = 0;  // both polarities (contiguous)
    __syncwarp();
    double m[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    int cnt[2] = {0, 0};
    for (int pol = 1; pol >= 0 && ok; --pol) {  // + first like the reference (sums are exact integers anyway)
        const ProbDesc d = a.prob[2 * w + pol];
        const int nk = a.hdr[2 * w + pol].n_kept;
        const KeptCluster *kt = a.ktab + (size_t) (2 * w + pol) * a.max_k;
        const uint32_t *pts = a.pts[pol] + d.off;
        const int32_t *lab = a.labels[pol] + d.off;
        for (int i = lane; i < d.n; i += 32) {
            const uint32_t p = pts[i];
            const double dx = (double) ECB_PIX_X(p) - ip[0], dy = (double) ECB_PIX_Y(p) - ip[1];
            const double d2 = dx * dx + dy * dy;
            if (!(d2 < R2)) continue;
            const double distance = sqrt(d2);
            int idx = 0;
            if (dx >= 0 && dy >= 0) idx = 0;
            else if (dx >= 0 && dy <= 0) idx = 1;
            else if (dx <= 0 && dy <= 0) idx = 2;
            else if (dx <= 0 && dy >= 0) idx = 3;
            const double rq = idx == 0 ? radius[0] : idx == 1 ? radius[1] : idx == 2 ? radius[2] : radius[3];
            if (!(fabs(distance - rq) <= a.thr)) continue;
            const int32_t l = lab[i];
            if (l < 0) continue;
            int lo = 0, hi = nk;  // kept clusters are listed in ascending raw id
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (kt[mid].raw_id < l) lo = mid + 1; else hi = mid;
            }
            if (lo < nk && kt[lo].raw_id == l) atomicOr(&mask[pol][lo >> 5], 1u << (lo & 31));
        }
        __syncwarp();
        for (int k = lane; k < nk; k += 32)
            if ((mask[pol][k >> 5] >> (k & 31)) & 1u) {
                cnt[pol] += kt[k].size;
#pragma unroll
                for (int q = 0; q < 9; ++q) m[q] += kt[k].m[q];
            }
    }
#pragma unroll
    for (int q = 0; q < 9; ++q) m[q] = warp_sum(m[q]);
    for (int pol = 0; pol < 2; ++pol)
        for (int off = 16; off > 0; off >>= 1) cnt[pol] += __shfl_xor_sync(0xffffffffu, cnt[pol], off);
    if (cnt[0] < 5 || cnt[1] < 5) ok = false;  // :558-561
    double cx = 0, cy = 0, r = -1;
    if (ok) {
        fit_from_moments(m, (double) (cnt[0] + cnt[1]), cx, cy, r);
        // median of the four quadrant radii = what std::nth_element leaves in slot 2 (:568)
        double s0 = radius[0], s1 = radius[1], s2 = radius[2], s3 = radius[3], t;
        if (s0 > s1) { t = s0; s0 = s1; s1 = t; }
        if (s2 > s3) { t = s2; s2 = s3; s3 = t; }
        if (s0 > s2) { t = s0; s0 = s2; s2 = t; }
        if (s1 > s3) { t = s1; s1 = s3; s3 = t; }
        if (s1 > s2) { t = s1; s1 = s2; s2 = t; }
        const double ex = cx - ip[0], ey = cy - ip[1];
        if (sqrt(ex * ex + ey * ey) > 2 * a.thr || fabs(r - s2) > 1.5 * a.thr) ok = false;  // :570-574
    }
    if (lane == 0) {
        o[0] = ok ? cx : 0.0;
        o[1] = ok ? cy : 0.0;
        o[2] = ok ? r : -1.0;
    }
}

// batched fit of explicit point sets: one warp per set (ecb_fit_circles)
__global__ void k_fit(const double *__restrict__ xy, const int64_t *__restrict__ off, int n_sets, double *__restrict__ out) {
    const int set = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (set >= n_sets) return;
    const int64_t b = off[set], e = off[set + 1];
    double m[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int64_t i = b + lane; i < e; i += 32) {
        const double x = xy[2 * i], y = xy[2 * i + 1];
        const double xx = x * x, yy = y * y, xyv = x * y;
        m[0] += x;
        m[1] += y;
        m[2] += xx;
        m[3] += yy;
        m[4] += xyv;
        m[5] += xx * x;
        m[6] += yy * y;
        m[7] += xyv * y;
        m[8] += x * xyv;
    }
#pragma unroll
    for (int q = 0; q < 9; ++q) m[q] = warp_sum(m[q]);
    if (lane == 0) {
        double cx, cy, r;
        fit_from_moments(m, (double) (e - b), cx, cy, r);
        out[3 * set] = cx;
        out[3 * set + 1] = cy;
        out[3 * set + 2] = r;
    }
}

}  // namespace

template <bool LANE>
static void (*direct_pair_kernel(bool fit, bool small_km))(const PairArgs) {
    return fit ? (small_km ? k_pair<true, true, false, ECB_PAIR_KM, LANE> : k_pair<true, true, false, KNN_MAX, LANE>)
               : k_pair<true, false, false, KNN_MAX, LANE>;
}

int ecb_launch_pair(ecb_ctx *ctx, PairArgs &a) {
    if (a.n_win <= 0) return ECB_OK;
    // kept-cluster tables: 44 bytes per entry, in shared memory unless there are very many kept clusters; member pixels are
    // staged in shared memory as well when both polarities of the largest window fit next to the tables
    const size_t tab = (((size_t) a.max_k * 44) + 15) & ~(size_t) 15;
    const size_t pix = (size_t) 2 * a.smem_cap * 4;
    const size_t cap = 96 * 1024;
    const bool gt = tab > cap;
    const bool direct = !gt && a.smem_cap > 0 && tab + pix <= cap;
    const size_t smem = gt ? 0 : tab + (direct ? pix : 0);
    const bool lane = direct && a.smem_cap <= PAIR_LANE_MAX_POINTS;
    const bool small_km = ECB_PAIR_KM4 && a.knn_num <= ECB_PAIR_KM;
    void (*kern)(const PairArgs) =
        gt ? (a.fit_circle ? k_pair<false, true, true, KNN_MAX, false> : k_pair<false, false, true, KNN_MAX, false>)
           : direct ? (lane ? direct_pair_kernel<true>(a.fit_circle, small_km) : direct_pair_kernel<false>(a.fit_circle, small_km))
                    : (a.fit_circle ? k_pair<false, true, false, KNN_MAX, false> : k_pair<false, false, false, KNN_MAX, false>);
    const int nt = lane ? PAIR_LANE_THREADS : PAIR_THREADS;
    ECB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) cap)  /* constant: race-free */);
    int grid = a.n_win < ctx->sm_count * 8 ? a.n_win : ctx->sm_count * 8;
    if (a.win_counter) {  // dynamic hand-out: the resident CTAs
        int per_sm = 0;
        ECB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nt, smem));
        grid = std::min(a.n_win, ctx->sm_count * std::max(per_sm, 1));
    }
    a.gtab = nullptr;
    a.gtab_stride = 0;
    if (gt) {
        a.gtab_stride = tab / 8;
        int rc = ecb_reserve(ctx, ctx->pair_tab, (size_t) grid * tab);
        if (rc) return rc;
        a.gtab = (double *) ctx->pair_tab.p;
    }
    ECB_PROF_BEGIN(ctx, ECB_STAGE_PAIR);
    kern<<<grid, nt, smem, ctx->stream>>>(a);
    ECB_PROF_END(ctx, ECB_STAGE_PAIR);
    ECB_LAUNCHED(ctx);
    return ecb_check(ctx, cudaGetLastError(), "k_pair launch");
}

int ecb_launch_fit(ecb_ctx *ctx, const double *d_xy, const int64_t *d_off, int n_sets, double *d_out) {
    if (n_sets <= 0) return ECB_OK;
    const int thr = 128;
    k_fit<<<(n_sets * 32 + thr - 1) / thr, thr, 0, ctx->stream>>>(d_xy, d_off, n_sets, d_out);
    ECB_LAUNCHED(ctx);
    return ecb_check(ctx, cudaGetLastError(), "k_fit launch");
}

int ecb_launch_rectify(ecb_ctx *ctx, const int32_t *d_win, int n_frames, int n_feat, const double *d_img, double *d_out,
                       const PairArgs &pa, const int32_t *const labels[2], double thr) {
    if (n_frames <= 0 || n_feat <= 0) return ECB_OK;
    RectifyArgs a;
    a.win = d_win;
    a.n_frames = n_frames;
    a.n_feat = n_feat;
    a.img = d_img;
    a.out = d_out;
    a.prob = pa.prob;
    a.hdr = pa.hdr;
    a.ktab = pa.ktab;
    for (int p = 0; p < 2; ++p) {
        a.pts[p] = pa.pts[p];
        a.labels[p] = labels[p];
    }
    a.max_k = pa.max_k;
    a.W = ctx->width;
    a.H = ctx->height;
    a.thr = thr;
    const int items = n_frames * n_feat;
    const size_t smem = (size_t) RECT_WARPS * 2 * ((a.max_k + 31) / 32) * 4;
    if (smem > 200 * 1024) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "rectify: %d kept clusters per window", a.max_k);
    ECB_CUDA(ctx, cudaFuncSetAttribute(k_rectify, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    k_rectify<<<(items + RECT_WARPS - 1) / RECT_WARPS, RECT_WARPS * 32, smem, ctx->stream>>>(a);
    ECB_LAUNCHED(ctx);
    return ecb_check(ctx, cudaGetLastError(), "k_rectify launch");
}
