// General DBSCAN path — DBSCAN<T,Float>::Run (dbscan/include/dbscan.h:115-265) for ANY input the reference accepts:
// non-integer coordinates, duplicate points, any eps (also 0 and negative), dim 1..ECB_GH_MAXD, any extent.  The sensor-plane
// bitmap kernel (ecb_cluster.cu) stays the fast path for what the calibration front end produces (distinct integer pixels,
// 1 <= eps <= 15); everything else lands here instead of being refused.
//
//   1. grid hash: cell = floor((p - min) / h) per axis, h = |eps| (1 + 2^-16) (two points within eps can never be more than
//      one cell apart, also after rounding); key = (problem, cell_{dim-1}, .., cell_0) packed into 64 bits; LSD radix sort
//      of (key, index) pairs written here (8-bit digits, stable, warp-match ranking); the 3^(dim-1) cell rows around a
//      point are contiguous ranges of the sorted array, found by binary search.  If the keys of a batch do not fit 64 bits
//      (or dim > 3) the candidate range of a point is its whole problem (brute force) — slower, same results.
//   2. neighbour test exactly as find_nearest evaluates it (kdtree.cpp:155-159): dist_sq accumulated in axis order from
//      rounded differences, no FMA contraction, compared with SQ(range).
//   3. what the kd query MISSES (kdtree.cpp:166-171: the far child is entered only if fabs(dx) < range, strictly): a pair can
//      only be lost if |fl(p[d] - q[d])| >= eps on some axis although dist_sq <= eps^2 ("boundary pair": integer grids with
//      integer eps, duplicates of such points, rounding slivers).  For those — and only those — the query is replayed on the
//      ancestor chain of p in the emulated tree: p is found iff for every ancestor A on whose far side (w.r.t. q) p hangs,
//      fabs(q[dir_A] - A[dir_A]) < eps.  The tree is the reference's: sequential insertion in pid order (kdtree.cpp:106-146),
//      emulated level-synchronously (one launch per tree level; atomicMin on the child slots decides who a slot belongs to).
//      It is only built when a batch has boundary pairs or ordered member lists are requested.
//   4. core <=> #found neighbours (self excluded by index, duplicates count) >= minPts (dbscan.h:150-151,218,244-247);
//      lock-free union-find over mutual core-core edges; one-way edges by min-label propagation; cluster id = rank of the
//      seed pid; non-core points are Noise — the same set formulation as ecb_cluster.cu (SURVEY Appendix A).
//   5. ordered `Clusters` (BFS pop order): k_bfs_order_general (ecb_bfs.cu) walks the same emulated tree.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "ecb_cluster.cuh"

namespace {

constexpr int GH_THREADS = 256;
constexpr int RS_ITEMS = 8;                      // keys per thread of the radix sort
constexpr int RS_TILE = GH_THREADS * RS_ITEMS;   // keys per block
constexpr int GH_MAXR = 9;                       // 3^(3-1) cell rows

struct GhArgs {
    const double *P;          // [n][dim] original order (pid order per problem)
    const double *SP;         // [n][dim] in sorted order (== P in brute-force mode)
    int dim;
    int64_t n;
    int n_prob;
    const int64_t *off;       // [n_prob + 1]
    const uint32_t *prob_of;  // [n] original index -> problem
    const uint32_t *sidx;     // sorted position -> original index
    const uint64_t *skey;     // sorted keys (grid mode)
    int grid;                 // 1: grid hash, 0: brute force
    int n_rows;               // candidate ranges per point
    uint32_t *nlo, *nhi;      // [n_rows][n]
    double eps, eps2;
    uint32_t min_pts;
    const uint4 *nodes;       // emulated kd-tree {left, right, parent, depth << 1 | side}, original indices; null: not built
    uint8_t *core;            // [n] by sorted position
    uint32_t *parent;         // union-find over sorted positions
    uint32_t *root;           // [n] root of every core point, ECB_NONE for non-core
    uint32_t *gmin, *glabel;  // [n] by root: lowest original index of the group / of everything that reaches it
    uint32_t *flags;          // [0] boundary pair seen, [1] label changed, [2] non-finite coordinate
};

// ---- order-preserving encoding of doubles for atomicMin / atomicMax --------------------------------------------------
__device__ __forceinline__ unsigned long long enc_d(double v) {
    const unsigned long long b = (unsigned long long) __double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
double dec_d(unsigned long long e) {
    const unsigned long long b = (e >> 63) ? (e & 0x7FFFFFFFFFFFFFFFull) : ~e;
    double v;
    memcpy(&v, &b, 8);
    return v;
}

__global__ void k_gh_prob_of(const int64_t *__restrict__ off, int n_prob, int64_t n, uint32_t *__restrict__ prob_of) {
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        int lo = 0, hi = n_prob;  // last problem with off <= i
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (off[mid] <= i) lo = mid; else hi = mid;
        }
        prob_of[i] = (uint32_t) lo;
    }
}

// per problem and axis: min and max coordinate (encoded), and a flag for NaN / Inf
__global__ void k_gh_minmax(const double *__restrict__ P, const uint32_t *__restrict__ prob_of, int64_t n, int dim,
                            unsigned long long *mn, unsigned long long *mx, uint32_t *flags) {
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        const uint32_t pb = prob_of[i];
        for (int d = 0; d < dim; ++d) {
            const double v = P[i * dim + d];
            if (!isfinite(v)) {
                flags[2] = 1;
                continue;
            }
            const unsigned long long e = enc_d(v);
            // neighbouring threads mostly belong to the same problem: test before the atomic
            if (e < mn[(size_t) pb * dim + d]) atomicMin(&mn[(size_t) pb * dim + d], e);
            if (e > mx[(size_t) pb * dim + d]) atomicMax(&mx[(size_t) pb * dim + d], e);
        }
    }
}

struct KeyLayout {
    int bits[3];   // bits per axis (cell + 1 stored, so that +-1 never wraps)
    int shift[3];
    int pshift;    // problem index above the cells
    double h;      // cell size
};

__device__ __forceinline__ uint64_t cell_of(double v, double mn, double h) {
    // floor((v - min) / h): plain IEEE operations, monotone in v
    return (uint64_t) floor(__ddiv_rn(__dsub_rn(v, mn), h)) + 1ull;
}

__global__ void k_gh_keys(const double *__restrict__ P, const uint32_t *__restrict__ prob_of, const double *__restrict__ pmin,
                          int64_t n, int dim, KeyLayout kl, uint64_t *__restrict__ key, uint32_t *__restrict__ idx) {
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        const uint32_t pb = prob_of[i];
        uint64_t k = (uint64_t) pb << kl.pshift;
        for (int d = 0; d < dim; ++d) k |= cell_of(P[i * dim + d], pmin[(size_t) pb * dim + d], kl.h) << kl.shift[d];
        key[i] = k;
        idx[i] = (uint32_t) i;
    }
}

// ---- LSD radix sort of (key, index) pairs, 8 bits per pass -------------------------------------------------------------
__global__ void __launch_bounds__(GH_THREADS) k_rs_hist(const uint64_t *__restrict__ key, int64_t n, int shift,
                                                         uint32_t *__restrict__ hist, int nblk) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t) blockIdx.x * RS_TILE;
    for (int v = 0; v < RS_ITEMS; ++v) {
        const int64_t i = base + v * GH_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&h[(key[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(size_t) threadIdx.x * nblk + blockIdx.x] = h[threadIdx.x];
}

// exclusive scan of m words by one block (in place); total -> *total if non-null
__global__ void __launch_bounds__(1024) k_scan_single(uint32_t *a, int64_t m, uint32_t *total) {
    __shared__ uint32_t ws[33];
    uint32_t carry = 0;
    for (int64_t b = 0; b < m; b += 1024) {
        const int64_t i = b + threadIdx.x;
        const uint32_t v = i < m ? a[i] : 0;
        uint32_t tot;
        const uint32_t ex = block_excl_scan(v, ws, &tot);
        if (i < m) a[i] = carry + ex;
        carry += tot;
    }
    if (total && threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(GH_THREADS) k_rs_scatter(const uint64_t *__restrict__ key, const uint32_t *__restrict__ idx,
                                                            uint64_t *__restrict__ key_out, uint32_t *__restrict__ idx_out,
                                                            int64_t n, int shift, const uint32_t *__restrict__ hist, int nblk) {
    __shared__ uint32_t whist[GH_THREADS / 32][256];
    __shared__ uint32_t gbase[256];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < (GH_THREADS / 32) * 256; i += GH_THREADS) (&whist[0][0])[i] = 0;
    __syncthreads();
    // warp w owns the contiguous keys [base + w * 256, +256): item v of lane l is key w*256 + v*32 + l  (stable order)
    const int64_t base = (int64_t) blockIdx.x * RS_TILE + w * (32 * RS_ITEMS);
    uint64_t k[RS_ITEMS];
    uint32_t rk[RS_ITEMS];
#pragma unroll
    for (int v = 0; v < RS_ITEMS; ++v) {
        const int64_t i = base + v * 32 + lane;
        const bool ok = i < n;
        k[v] = ok ? key[i] : 0;
        const uint32_t d = ok ? (uint32_t) ((k[v] >> shift) & 255u) : 0xFFFFFFFFu;
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const int leader = __ffs(peers) - 1;
        uint32_t pre = 0;
        if (ok && lane == leader) {
            pre = whist[w][d];
            whist[w][d] = pre + __popc(peers);
        }
        pre = __shfl_sync(0xffffffffu, pre, leader);
        rk[v] = pre + __popc(peers & ((1u << lane) - 1u));
        __syncwarp();
    }
    __syncthreads();
    {
        const int d = threadIdx.x;  // one digit per thread: exclusive scan over the warps
        uint32_t run = 0;
#pragma unroll
        for (int ww = 0; ww < GH_THREADS / 32; ++ww) {
            const uint32_t t = whist[ww][d];
            whist[ww][d] = run;
            run += t;
        }
        gbase[d] = hist[(size_t) d * nblk + blockIdx.x];
    }
    __syncthreads();
#pragma unroll
    for (int v = 0; v < RS_ITEMS; ++v) {
        const int64_t i = base + v * 32 + lane;
        if (i < n) {
            const uint32_t d = (uint32_t) ((k[v] >> shift) & 255u);
            const uint32_t dst = gbase[d] + whist[w][d] + rk[v];
            key_out[dst] = k[v];
            idx_out[dst] = idx[i];
        }
    }
}

// ---- sorted-order helpers ------------------------------------------------------------------------------------------------
__global__ void k_gh_gather(const double *__restrict__ P, const uint32_t *__restrict__ sidx, int64_t n, int dim,
                            double *__restrict__ SP) {
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        const size_t o = sidx[i];
        for (int d = 0; d < dim; ++d) SP[i * dim + d] = P[o * dim + d];
    }
}

__device__ __forceinline__ uint32_t lower_bound_key(const uint64_t *k, int64_t n, uint64_t v) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (k[mid] < v) lo = mid + 1; else hi = mid;
    }
    return (uint32_t) lo;
}

// candidate ranges of every sorted point: the 3^(dim-1) rows of cells (c0-1 .. c0+1) around it
__global__ void k_gh_ranges(GhArgs a, KeyLayout kl) {
    const int64_t n = a.n;
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        const uint64_t k = a.skey[i];
        const uint64_t m0 = (1ull << kl.bits[0]) - 1ull;
        const uint64_t c0 = (k >> kl.shift[0]) & m0;
        for (int r = 0; r < a.n_rows; ++r) {
            // row offsets of the higher axes: r = (o1 + 1) + 3 (o2 + 1)
            uint64_t kk = k & ~(m0 << kl.shift[0]);
            int rr = r;
            for (int d = 1; d < a.dim; ++d) {
                const int o = rr % 3 - 1;
                rr /= 3;
                kk += (uint64_t) (int64_t) o << kl.shift[d];  // cells are stored + 1 and have a spare value on top: no wrap
            }
            const uint64_t klo = kk | ((c0 - 1ull) << kl.shift[0]), khi = kk | ((c0 + 1ull) << kl.shift[0]);
            a.nlo[(size_t) r * n + i] = lower_bound_key(a.skey, n, klo);
            a.nhi[(size_t) r * n + i] = lower_bound_key(a.skey, n, khi + 1ull);
        }
    }
}

__global__ void k_gh_iota(uint32_t *idx, int64_t n) {
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) idx[i] = (uint32_t) i;
}

__global__ void k_gh_ranges_brute(GhArgs a) {
    const int64_t n = a.n;
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        const uint32_t pb = a.prob_of[i];
        a.nlo[i] = (uint32_t) a.off[pb];
        a.nhi[i] = (uint32_t) a.off[pb + 1];
    }
}

// ---- the neighbour relation -------------------------------------------------------------------------------------------------
// dist_sq <= SQ(range) with the reference's operation order; *boundary = some axis has |fl(p - q)| >= eps
__device__ __forceinline__ bool gh_near(const double *p, const double *q, int dim, double eps, double eps2, bool *boundary) {
    double d2 = 0.0;
    bool b = false;
    for (int d = 0; d < dim; ++d) {
        const double e = __dsub_rn(p[d], q[d]);
        d2 = __dadd_rn(d2, __dmul_rn(e, e));
        b |= !(fabs(e) < eps);
    }
    *boundary = b;
    return d2 <= eps2;
}

// does kd_nearest_range at q (original coordinates) reach the node of p?  Replays the pruning rule on p's ancestors.
__device__ bool gh_kd_finds(const GhArgs &a, const double *q, uint32_t p) {
    uint4 nd = a.nodes[p];
    while (nd.z != ECB_NONE) {
        const uint32_t A = nd.z;
        const int side = (int) (nd.w & 1u);
        const int dir = (int) (((nd.w >> 1) - 1u) % (uint32_t) a.dim);  // depth of A = depth of the child - 1
        const double dx = __dsub_rn(q[dir], a.P[(size_t) A * a.dim + dir]);
        const bool near_left = dx <= 0.0;
        if (near_left != (side == 0) && !(fabs(dx) < a.eps)) return false;  // p hangs on the far side and it is pruned
        nd = a.nodes[A];
    }
    return true;
}

// neighbour count and core flag.  exact = 0: boundary pairs are counted as found and reported in flags[0] (the caller then
// builds the tree and runs the pass again with exact = 1).
__global__ void __launch_bounds__(GH_THREADS) k_gh_count(GhArgs a, int exact) {
    const int64_t n = a.n;
    const int dim = a.dim;
    bool saw_boundary = false;
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        double q[ECB_GH_MAXD];
        for (int d = 0; d < dim; ++d) q[d] = a.SP[i * dim + d];
        uint32_t cnt = 0;
        for (int r = 0; r < a.n_rows; ++r) {
            const uint32_t lo = a.nlo[(size_t) r * n + i], hi = a.nhi[(size_t) r * n + i];
            for (uint32_t j = lo; j < hi; ++j) {
                if (j == (uint32_t) i) continue;  // self is excluded by index (dbscan.h:218); duplicates are neighbours
                bool bnd;
                if (!gh_near(a.SP + (size_t) j * dim, q, dim, a.eps, a.eps2, &bnd)) continue;
                if (bnd) {
                    if (!exact)
                        saw_boundary = true;
                    else if (!gh_kd_finds(a, q, a.sidx[j]))
                        continue;
                }
                ++cnt;
            }
        }
        a.core[i] = cnt >= a.min_pts;
        a.parent[i] = (uint32_t) i;
        a.root[i] = ECB_NONE;
        a.gmin[i] = ECB_NONE;
    }
    if (saw_boundary) a.flags[0] = 1;
}

__device__ __forceinline__ uint32_t gh_find_root(volatile uint32_t *parent, uint32_t x) {
    uint32_t p = parent[x];
    while (p != x) {
        const uint32_t g = parent[p];
        if (g != p) parent[x] = g;  // path halving (benign race: only ever points to an ancestor)
        x = p;
        p = g;
    }
    return x;
}

__device__ __forceinline__ void gh_unite(uint32_t *parent, uint32_t x, uint32_t y) {
    for (;;) {
        x = gh_find_root(parent, x);
        y = gh_find_root(parent, y);
        if (x == y) return;
        if (x < y) {
            const uint32_t t = x;
            x = y;
            y = t;
        }
        if (atomicCAS(&parent[x], x, y) == x) return;
    }
}

// union-find over MUTUAL core-core edges (every unordered pair once: j > i)
__global__ void __launch_bounds__(GH_THREADS) k_gh_union(GhArgs a) {
    const int64_t n = a.n;
    const int dim = a.dim;
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        if (!a.core[i]) continue;
        double q[ECB_GH_MAXD];
        for (int d = 0; d < dim; ++d) q[d] = a.SP[i * dim + d];
        for (int r = 0; r < a.n_rows; ++r) {
            const uint32_t lo = max(a.nlo[(size_t) r * n + i], (uint32_t) i + 1u), hi = a.nhi[(size_t) r * n + i];
            for (uint32_t j = lo; j < hi; ++j) {
                if (!a.core[j]) continue;
                bool bnd;
                const double *pj = a.SP + (size_t) j * dim;
                if (!gh_near(pj, q, dim, a.eps, a.eps2, &bnd)) continue;
                if (bnd && a.nodes && !(gh_kd_finds(a, q, a.sidx[j]) && gh_kd_finds(a, pj, a.sidx[i]))) continue;
                gh_unite(a.parent, (uint32_t) i, j);
            }
        }
    }
}

__global__ void k_gh_flatten(GhArgs a) {
    const int64_t n = a.n;
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        if (!a.core[i]) continue;
        const uint32_t r = gh_find_root(a.parent, (uint32_t) i);
        a.root[i] = r;
        atomicMin(&a.gmin[r], a.sidx[i]);
    }
}

__global__ void k_gh_copy_u32(const uint32_t *__restrict__ src, uint32_t *__restrict__ dst, int64_t n) {
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) dst[i] = src[i];
}

// one-way edges (query at i finds j, the reverse is pruned): the label of i's group flows to j's group
__global__ void __launch_bounds__(GH_THREADS) k_gh_propagate(GhArgs a) {
    const int64_t n = a.n;
    const int dim = a.dim;
    bool changed = false;
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        const uint32_t ri = a.root[i];
        if (ri == ECB_NONE) continue;
        double q[ECB_GH_MAXD];
        for (int d = 0; d < dim; ++d) q[d] = a.SP[i * dim + d];
        for (int r = 0; r < a.n_rows; ++r) {
            const uint32_t lo = a.nlo[(size_t) r * n + i], hi = a.nhi[(size_t) r * n + i];
            for (uint32_t j = lo; j < hi; ++j) {
                const uint32_t rj = a.root[j];
                if (rj == ECB_NONE || rj == ri) continue;
                bool bnd;
                if (!gh_near(a.SP + (size_t) j * dim, q, dim, a.eps, a.eps2, &bnd) || !bnd) continue;
                if (!gh_kd_finds(a, q, a.sidx[j])) continue;
                const uint32_t li = ((volatile uint32_t *) a.glabel)[ri];
                if (li < atomicMin(&a.glabel[rj], li)) changed = true;
            }
        }
    }
    if (changed) a.flags[1] = 1;
}

// a group is a seed iff nothing smaller reached it; the seed pid is its own lowest member
__global__ void k_gh_seeds(GhArgs a, uint32_t *seedflag) {
    const int64_t n = a.n;
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x)
        if (a.root[i] == (uint32_t) i && a.glabel[i] == a.gmin[i]) seedflag[a.gmin[i]] = 1u;
}

__global__ void k_gh_labels(GhArgs a, const uint32_t *__restrict__ seedpref, int32_t *__restrict__ labels) {
    const int64_t n = a.n;
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        const uint32_t o = a.sidx[i], r = a.root[i];
        int32_t lab = -1;
        if (r != ECB_NONE) lab = (int32_t) (seedpref[a.glabel[r]] - seedpref[a.off[a.prob_of[o]]]);
        labels[o] = lab;
    }
}

__global__ void k_gh_headers(const int64_t *__restrict__ off, int n_prob, const uint32_t *__restrict__ seedpref, ProbDesc *pd,
                             ProbHdr *hdr) {
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_prob; k += gridDim.x * blockDim.x) {
        ProbDesc d;
        d.off = off[k];
        d.n = (int32_t) (off[k + 1] - off[k]);
        d.pol = 0;
        d.x0 = d.y0 = d.pad0 = d.pad1 = 0;
        pd[k] = d;
        ProbHdr h;
        h.n_clusters = (int32_t) (seedpref[off[k + 1]] - seedpref[off[k]]);
        h.n_kept = 0;
        h.n_core = 0;
        h.status = 0;
        hdr[k] = h;
    }
}

// ---- kd insertion emulation: one launch per tree level ----------------------------------------------------------------------
// state[i] = node the point currently stands at | side it wants to descend to << 31; ECB_NONE once inserted.
__global__ void k_kd_init(const int64_t *__restrict__ off, const uint32_t *__restrict__ prob_of, int64_t n, uint4 *nodes,
                          uint32_t *state) {
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        const uint32_t root = (uint32_t) off[prob_of[i]];
        nodes[i] = make_uint4(ECB_NONE, ECB_NONE, ECB_NONE, 0u);  // the root keeps depth 0, no parent
        state[i] = (uint32_t) i == root ? ECB_NONE : (root | 0x40000000u);  // bit 30: no pending slot yet
    }
}

// round r: resolve the slot claimed in round r-1 (the winner is inserted there, the others step down to it), then claim a
// child slot of the node now stood at (a node of depth r, split axis r % dim: pos[dir] < node.pos[dir] -> left)
__global__ void k_kd_round(const double *__restrict__ P, int64_t n, int dim, int round, uint4 *nodes, uint32_t *state,
                           uint32_t *flag) {
    uint32_t *slots = reinterpret_cast<uint32_t *>(nodes);
    const int dir = round % dim;
    bool any = false;
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        uint32_t st = state[i];
        if (st == ECB_NONE) continue;
        uint32_t cur = st & 0x3FFFFFFFu;
        if (!(st & 0x40000000u)) {
            const uint32_t side = st >> 31;
            const uint32_t c = slots[4 * (size_t) cur + side];
            if (c == (uint32_t) i) {
                nodes[i].z = cur;
                nodes[i].w = ((uint32_t) round << 1) | side;  // depth of i = round
                state[i] = ECB_NONE;
                continue;
            }
            cur = c;
        }
        const uint32_t side = P[i * dim + dir] < P[(size_t) cur * dim + dir] ? 0u : 1u;
        atomicMin(&slots[4 * (size_t) cur + side], (uint32_t) i);
        state[i] = cur | (side << 31);
        any = true;
    }
    if (any) *flag = 1;
}

int grid_for(const ecb_ctx *ctx, int64_t n) {
    const int64_t need = (n + GH_THREADS - 1) / GH_THREADS;
    return (int) std::max<int64_t>(1, std::min<int64_t>(need, (int64_t) ctx->sm_count * 16));
}

}  // namespace

#define GH_LAUNCH(ctx, what)                                             \
    do {                                                                 \
        ECB_LAUNCHED(ctx);                                               \
        int _rc = ecb_check((ctx), cudaGetLastError(), what " launch");  \
        if (_rc) return _rc;                                             \
    } while (0)

// Device-wide exclusive scan of n words (in place) = per-tile sums, scan of the sums, per-tile scan.
namespace {
__global__ void __launch_bounds__(GH_THREADS) k_scan_tiles(const uint32_t *__restrict__ a, int64_t n, uint32_t *__restrict__ sums) {
    __shared__ uint32_t ws[33];
    const int64_t base = (int64_t) blockIdx.x * RS_TILE + (int64_t) threadIdx.x * RS_ITEMS;
    uint32_t s = 0;
    for (int v = 0; v < RS_ITEMS; ++v)
        if (base + v < n) s += a[base + v];
    uint32_t tot;
    block_excl_scan(s, ws, &tot);
    if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}
__global__ void __launch_bounds__(GH_THREADS) k_scan_apply(uint32_t *a, int64_t n, const uint32_t *__restrict__ sums) {
    __shared__ uint32_t ws[33];
    const int64_t base = (int64_t) blockIdx.x * RS_TILE + (int64_t) threadIdx.x * RS_ITEMS;
    uint32_t v[RS_ITEMS], s = 0;
    for (int k = 0; k < RS_ITEMS; ++k) {
        v[k] = base + k < n ? a[base + k] : 0;
        s += v[k];
    }
    uint32_t tot;
    uint32_t ex = block_excl_scan(s, ws, &tot) + sums[blockIdx.x];
    for (int k = 0; k < RS_ITEMS; ++k) {
        if (base + k < n) a[base + k] = ex;
        ex += v[k];
    }
}
}  // namespace

static int gh_scan(ecb_ctx *ctx, uint32_t *a, int64_t n, uint32_t *sums) {
    const int nblk = (int) ((n + RS_TILE - 1) / RS_TILE);
    k_scan_tiles<<<nblk, GH_THREADS, 0, ctx->stream>>>(a, n, sums);
    GH_LAUNCH(ctx, "k_scan_tiles");
    k_scan_single<<<1, 1024, 0, ctx->stream>>>(sums, nblk, nullptr);
    GH_LAUNCH(ctx, "k_scan_single");
    k_scan_apply<<<nblk, GH_THREADS, 0, ctx->stream>>>(a, n, sums);
    GH_LAUNCH(ctx, "k_scan_apply");
    return ECB_OK;
}

// Sorts (key, idx) by the low `bits` bits of key; the result ends in key[*res] / idx[*res] (ping-pong buffers 0 / 1).
// Declared in ecb_common.cuh (the residual report of ecb_cost.cu sorts records by group with it).
int gh_radix_sort(ecb_ctx *ctx, uint64_t *key[2], uint32_t *idx[2], int64_t n, int bits, uint32_t *hist, int *res) {
    const int nblk = (int) ((n + RS_TILE - 1) / RS_TILE);
    int cur = 0;
    for (int shift = 0; shift < bits; shift += 8) {
        k_rs_hist<<<nblk, GH_THREADS, 0, ctx->stream>>>(key[cur], n, shift, hist, nblk);
        GH_LAUNCH(ctx, "k_rs_hist");
        k_scan_single<<<1, 1024, 0, ctx->stream>>>(hist, (int64_t) 256 * nblk, nullptr);
        GH_LAUNCH(ctx, "k_scan_single");
        k_rs_scatter<<<nblk, GH_THREADS, 0, ctx->stream>>>(key[cur], idx[cur], key[cur ^ 1], idx[cur ^ 1], n, shift, hist, nblk);
        GH_LAUNCH(ctx, "k_rs_scatter");
        cur ^= 1;
    }
    *res = cur;
    return ECB_OK;
}

size_t gh_radix_hist_bytes(int64_t n) { return (size_t) 256 * (size_t) ((n + RS_TILE - 1) / RS_TILE) * 4; }

static int bits_for(uint64_t v) {  // bits needed to store values 0..v
    int b = 1;
    while (b < 64 && (v >> b)) ++b;
    return b;
}

// The general DBSCAN of a batch of problems.  pts: host [total][dim]; labels (host, may be null), n_clusters (host, may be
// null); ordered: cluster_sizes / members (host) like ecb_dbscan_run_batch_ordered.
int ecb_dbscan_general(ecb_ctx *ctx, const double *pts, int dim, const int64_t *offsets, int n_problems, double eps,
                       uint32_t min_pts, int32_t *labels, int32_t *n_clusters, int32_t *cluster_sizes, uint32_t *members) {
    if (dim < 1) return ecb_fail(ctx, ECB_FAILED, "dim < 1 (dbscan.h:122)");
    if (dim > ECB_GH_MAXD) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "dbscan dim %d > %d", dim, ECB_GH_MAXD);
    if (!(eps == eps)) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "dbscan eps is NaN");
    const int64_t n = offsets[n_problems];
    for (int k = 0; k < n_problems; ++k) {
        if (offsets[k + 1] - offsets[k] < 1) return ecb_fail(ctx, ECB_FAILED, "problem %d: V->size() < 1 (dbscan.h:121)", k);
        if (offsets[k + 1] - offsets[k] >= (1ll << 21))
            return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "problem %d: more than 2^21 - 1 points", k);
    }
    if (n >= 0x3FFFFFFFll) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "batch of %lld points", (long long) n);
    const bool ordered = cluster_sizes && members;
    int rc;
    DevBuf *B = ctx->gh;
    enum { B_P, B_SP, B_OFF, B_PROB, B_MM, B_PMIN, B_KEY0, B_KEY1, B_IDX0, B_IDX1, B_HIST, B_NLO, B_NHI, B_CORE, B_PARENT,
           B_ROOT, B_GMIN, B_GLABEL, B_FLAGS, B_NODES, B_STATE, B_SEED, B_SUMS, B_LABELS, B_PD, B_HDR, B_COUNT };
    static_assert(B_COUNT <= ECB_GH_NBUF, "ctx->gh too small");
    const size_t un = (size_t) n;
    const int g = grid_for(ctx, n);
    cudaStream_t st = ctx->stream;
    if ((rc = ecb_reserve(ctx, B[B_P], un * dim * 8))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_OFF], (size_t) (n_problems + 1) * 8))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_PROB], un * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_MM], (size_t) n_problems * dim * 16))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_PMIN], (size_t) n_problems * dim * 8))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_FLAGS], 64))) return rc;
    ECB_CUDA(ctx, cudaMemcpyAsync(B[B_P].p, pts, un * dim * 8, cudaMemcpyHostToDevice, st));
    ECB_CUDA(ctx, cudaMemcpyAsync(B[B_OFF].p, offsets, (size_t) (n_problems + 1) * 8, cudaMemcpyHostToDevice, st));
    ECB_CUDA(ctx, cudaMemsetAsync(B[B_FLAGS].p, 0, 64, st));
    unsigned long long *mn = (unsigned long long *) B[B_MM].p, *mx = mn + (size_t) n_problems * dim;
    ECB_CUDA(ctx, cudaMemsetAsync(mn, 0xFF, (size_t) n_problems * dim * 8, st));
    ECB_CUDA(ctx, cudaMemsetAsync(mx, 0, (size_t) n_problems * dim * 8, st));
    const double *dP = (const double *) B[B_P].p;
    const int64_t *dOff = (const int64_t *) B[B_OFF].p;
    uint32_t *dProb = (uint32_t *) B[B_PROB].p, *dFlags = (uint32_t *) B[B_FLAGS].p;
    k_gh_prob_of<<<g, GH_THREADS, 0, st>>>(dOff, n_problems, n, dProb);
    GH_LAUNCH(ctx, "k_gh_prob_of");
    k_gh_minmax<<<g, GH_THREADS, 0, st>>>(dP, dProb, n, dim, mn, mx, dFlags);
    GH_LAUNCH(ctx, "k_gh_minmax");
    std::vector<unsigned long long> hmm((size_t) n_problems * dim * 2);
    uint32_t hflags[4];
    ECB_CUDA(ctx, cudaMemcpyAsync(hmm.data(), mn, hmm.size() * 8, cudaMemcpyDeviceToHost, st));
    ECB_CUDA(ctx, cudaMemcpyAsync(hflags, dFlags, 16, cudaMemcpyDeviceToHost, st));
    ECB_CUDA(ctx, cudaStreamSynchronize(st));
    if (hflags[2]) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "dbscan input holds NaN or infinite coordinates");

    // ---- grid layout: does (problem, cells) fit 64 bits? -----------------------------------------------------------
    KeyLayout kl;
    memset(&kl, 0, sizeof kl);
    const double aeps = fabs(eps);
    kl.h = aeps > 0.0 ? aeps * (1.0 + 1.0 / 65536.0) : 1.0;
    bool grid = dim <= 3 && std::isfinite(kl.h) && kl.h > 0.0;
    std::vector<double> pmin((size_t) n_problems * dim);
    int total_bits = 0;
    if (grid) {
        uint64_t maxc[3] = {0, 0, 0};
        for (int k = 0; k < n_problems && grid; ++k)
            for (int d = 0; d < dim; ++d) {
                const double lo = dec_d(hmm[(size_t) k * dim + d]), hi = dec_d(hmm[(size_t) n_problems * dim + (size_t) k * dim + d]);
                pmin[(size_t) k * dim + d] = lo;
                const double c = floor((hi - lo) / kl.h);
                if (!(c < 2147483648.0)) {  // rounding of the cell index would exceed the 2^-16 margin of h
                    grid = false;
                    break;
                }
                maxc[d] = std::max(maxc[d], (uint64_t) c);
            }
        if (grid) {
            int sh = 0;
            for (int d = 0; d < dim; ++d) {
                kl.bits[d] = bits_for(maxc[d] + 2);  // cells are stored + 1; one spare value on top
                kl.shift[d] = sh;
                sh += kl.bits[d];
            }
            kl.pshift = sh;
            total_bits = sh + (n_problems > 1 ? bits_for((uint64_t) n_problems - 1) : 0);
            if (total_bits > 63) grid = false;
        }
    }

    GhArgs a;
    memset(&a, 0, sizeof a);
    a.P = dP;
    a.dim = dim;
    a.n = n;
    a.n_prob = n_problems;
    a.off = dOff;
    a.prob_of = dProb;
    a.eps = eps;
    a.eps2 = eps * eps;
    a.min_pts = min_pts;
    a.grid = grid ? 1 : 0;
    a.flags = dFlags;
    a.n_rows = 1;
    if (grid)
        for (int d = 1; d < dim; ++d) a.n_rows *= 3;
    if ((rc = ecb_reserve(ctx, B[B_NLO], un * a.n_rows * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_NHI], un * a.n_rows * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_IDX0], un * 4))) return rc;
    a.nlo = (uint32_t *) B[B_NLO].p;
    a.nhi = (uint32_t *) B[B_NHI].p;
    if (grid) {
        const int nblk = (int) ((n + RS_TILE - 1) / RS_TILE);
        if ((rc = ecb_reserve(ctx, B[B_KEY0], un * 8))) return rc;
        if ((rc = ecb_reserve(ctx, B[B_KEY1], un * 8))) return rc;
        if ((rc = ecb_reserve(ctx, B[B_IDX1], un * 4))) return rc;
        if ((rc = ecb_reserve(ctx, B[B_HIST], (size_t) 256 * nblk * 4))) return rc;
        if ((rc = ecb_reserve(ctx, B[B_SP], un * dim * 8))) return rc;
        ECB_CUDA(ctx, cudaMemcpyAsync(B[B_PMIN].p, pmin.data(), pmin.size() * 8, cudaMemcpyHostToDevice, st));
        uint64_t *key[2] = {(uint64_t *) B[B_KEY0].p, (uint64_t *) B[B_KEY1].p};
        uint32_t *idx[2] = {(uint32_t *) B[B_IDX0].p, (uint32_t *) B[B_IDX1].p};
        k_gh_keys<<<g, GH_THREADS, 0, st>>>(dP, dProb, (const double *) B[B_PMIN].p, n, dim, kl, key[0], idx[0]);
        GH_LAUNCH(ctx, "k_gh_keys");
        int res = 0;
        if ((rc = gh_radix_sort(ctx, key, idx, n, total_bits, (uint32_t *) B[B_HIST].p, &res))) return rc;
        a.skey = key[res];
        a.sidx = idx[res];
        k_gh_gather<<<g, GH_THREADS, 0, st>>>(dP, a.sidx, n, dim, (double *) B[B_SP].p);
        GH_LAUNCH(ctx, "k_gh_gather");
        a.SP = (const double *) B[B_SP].p;
        k_gh_ranges<<<g, GH_THREADS, 0, st>>>(a, kl);
        GH_LAUNCH(ctx, "k_gh_ranges");
    } else {
        // brute force: the "sorted" order is the input order, the candidate range of a point is its whole problem
        uint32_t *idx0 = (uint32_t *) B[B_IDX0].p;
        k_gh_iota<<<g, GH_THREADS, 0, st>>>(idx0, n);
        GH_LAUNCH(ctx, "k_gh_iota");
        a.sidx = idx0;
        a.SP = dP;
        k_gh_ranges_brute<<<g, GH_THREADS, 0, st>>>(a);
        GH_LAUNCH(ctx, "k_gh_ranges_brute");
    }

    if ((rc = ecb_reserve(ctx, B[B_CORE], un))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_PARENT], un * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_ROOT], un * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_GMIN], un * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_GLABEL], un * 4))) return rc;
    a.core = (uint8_t *) B[B_CORE].p;
    a.parent = (uint32_t *) B[B_PARENT].p;
    a.root = (uint32_t *) B[B_ROOT].p;
    a.gmin = (uint32_t *) B[B_GMIN].p;
    a.glabel = (uint32_t *) B[B_GLABEL].p;

    // ---- neighbour counts; the tree only if a pair needs it -------------------------------------------------------
    bool need_tree = ordered;
    if (!need_tree) {
        k_gh_count<<<g, GH_THREADS, 0, st>>>(a, 0);
        GH_LAUNCH(ctx, "k_gh_count");
        ECB_CUDA(ctx, cudaMemcpyAsync(hflags, dFlags, 16, cudaMemcpyDeviceToHost, st));
        ECB_CUDA(ctx, cudaStreamSynchronize(st));
        need_tree = hflags[0] != 0;
    }
    if (need_tree) {
        if ((rc = ecb_reserve(ctx, B[B_NODES], un * 16))) return rc;
        if ((rc = ecb_reserve(ctx, B[B_STATE], un * 4))) return rc;
        uint4 *nodes = (uint4 *) B[B_NODES].p;
        uint32_t *state = (uint32_t *) B[B_STATE].p;
        k_kd_init<<<g, GH_THREADS, 0, st>>>(dOff, dProb, n, nodes, state);
        GH_LAUNCH(ctx, "k_kd_init");
        for (int round = 0;;) {
            // eight levels per host round trip; flags[4 + k] = "somebody is still walking after level k of this chunk"
            ECB_CUDA(ctx, cudaMemsetAsync(dFlags + 4, 0, 32, st));
            for (int k = 0; k < 8; ++k, ++round) {
                k_kd_round<<<g, GH_THREADS, 0, st>>>(dP, n, dim, round, nodes, state, dFlags + 4 + k);
                GH_LAUNCH(ctx, "k_kd_round");
            }
            uint32_t hf[8];
            ECB_CUDA(ctx, cudaMemcpyAsync(hf, dFlags + 4, 32, cudaMemcpyDeviceToHost, st));
            ECB_CUDA(ctx, cudaStreamSynchronize(st));
            if (!hf[7]) break;
        }
        a.nodes = nodes;
        k_gh_count<<<g, GH_THREADS, 0, st>>>(a, 1);
        GH_LAUNCH(ctx, "k_gh_count");
    }
    k_gh_union<<<g, GH_THREADS, 0, st>>>(a);
    GH_LAUNCH(ctx, "k_gh_union");
    k_gh_flatten<<<g, GH_THREADS, 0, st>>>(a);
    GH_LAUNCH(ctx, "k_gh_flatten");
    k_gh_copy_u32<<<g, GH_THREADS, 0, st>>>(a.gmin, a.glabel, n);
    GH_LAUNCH(ctx, "k_gh_copy_u32");
    if (a.nodes) {
        for (;;) {
            ECB_CUDA(ctx, cudaMemsetAsync(dFlags + 1, 0, 4, st));
            k_gh_propagate<<<g, GH_THREADS, 0, st>>>(a);
            GH_LAUNCH(ctx, "k_gh_propagate");
            ECB_CUDA(ctx, cudaMemcpyAsync(hflags, dFlags, 16, cudaMemcpyDeviceToHost, st));
            ECB_CUDA(ctx, cudaStreamSynchronize(st));
            if (!hflags[1]) break;
        }
    }
    // ---- seeds -> cluster ids ----------------------------------------------------------------------------------------------
    const int nblk1 = (int) ((n + 1 + RS_TILE - 1) / RS_TILE);
    if ((rc = ecb_reserve(ctx, B[B_SEED], (un + 1) * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_SUMS], (size_t) nblk1 * 4 + 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_LABELS], un * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_PD], (size_t) n_problems * sizeof(ProbDesc)))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_HDR], (size_t) n_problems * sizeof(ProbHdr)))) return rc;
    uint32_t *seed = (uint32_t *) B[B_SEED].p;
    ECB_CUDA(ctx, cudaMemsetAsync(seed, 0, (un + 1) * 4, st));
    k_gh_seeds<<<g, GH_THREADS, 0, st>>>(a, seed);
    GH_LAUNCH(ctx, "k_gh_seeds");
    if ((rc = gh_scan(ctx, seed, n + 1, (uint32_t *) B[B_SUMS].p))) return rc;
    int32_t *dLabels = (int32_t *) B[B_LABELS].p;
    k_gh_labels<<<g, GH_THREADS, 0, st>>>(a, seed, dLabels);
    GH_LAUNCH(ctx, "k_gh_labels");
    ProbDesc *pd = (ProbDesc *) B[B_PD].p;
    ProbHdr *hdr = (ProbHdr *) B[B_HDR].p;
    k_gh_headers<<<std::max(1, std::min(n_problems / 256 + 1, 1024)), 256, 0, st>>>(dOff, n_problems, seed, pd, hdr);
    GH_LAUNCH(ctx, "k_gh_headers");

    if (ordered) {
        if ((rc = ecb_reserve(ctx, ctx->db_scratch, un * 4))) return rc;
        if ((rc = ecb_reserve(ctx, ctx->bfs_key, un * 8))) return rc;
        if ((rc = ecb_reserve(ctx, ctx->bfs_items, un * sizeof(BfsItem) + 16))) return rc;
        if ((rc = ecb_reserve(ctx, ctx->bfs_front, un * 4))) return rc;
        if ((rc = ecb_reserve(ctx, ctx->bfs_tab, 3 * un * 4))) return rc;
        ECB_CUDA(ctx, cudaMemsetAsync(ctx->bfs_key.p, 0xFF, un * 8, st));
        ECB_CUDA(ctx, cudaMemsetAsync(ctx->bfs_items.p, 0, 16, st));
        uint32_t *csize = (uint32_t *) ctx->bfs_tab.p, *cseed = csize + un, *coff = cseed + un;
        BfsItem *items = (BfsItem *) ((char *) ctx->bfs_items.p + 16);
        if ((rc = ecb_launch_bfs_all_items(ctx, pd, hdr, n_problems, dLabels, csize, cseed, coff, items,
                                           (unsigned *) ctx->bfs_items.p, (int) un)))
            return rc;
        BfsArgs ba;
        memset(&ba, 0, sizeof ba);
        ba.items = items;
        ba.count = (const unsigned *) ctx->bfs_items.p;
        ba.max_items = (int) un;
        ba.prob = pd;
        for (int p = 0; p < 2; ++p) {
            ba.labels[p] = dLabels;
            ba.kd_nodes[p] = a.nodes;
            ba.members[p] = (uint32_t *) ctx->db_scratch.p;
            ba.scratch[p] = (uint32_t *) ctx->bfs_front.p;
            ba.key[p] = (unsigned long long *) ctx->bfs_key.p;
        }
        ba.init_keys = 0;
        ba.eps = eps;
        // the tree and the coordinates are indexed by ORIGINAL index; a problem's slice starts at its offset
        if ((rc = ecb_launch_bfs_general(ctx, ba, dP, dim))) return rc;
        ECB_CUDA(ctx, cudaMemcpyAsync(members, ctx->db_scratch.p, un * 4, cudaMemcpyDeviceToHost, st));
        ECB_CUDA(ctx, cudaMemcpyAsync(cluster_sizes, csize, un * 4, cudaMemcpyDeviceToHost, st));
    }
    std::vector<ProbHdr> hh((size_t) n_problems);
    if (labels) ECB_CUDA(ctx, cudaMemcpyAsync(labels, dLabels, un * 4, cudaMemcpyDeviceToHost, st));
    ECB_CUDA(ctx, cudaMemcpyAsync(hh.data(), hdr, (size_t) n_problems * sizeof(ProbHdr), cudaMemcpyDeviceToHost, st));
    ECB_CUDA(ctx, cudaStreamSynchronize(st));
    if (n_clusters)
        for (int k = 0; k < n_problems; ++k) n_clusters[k] = hh[(size_t) k].n_clusters;
    return ECB_OK;
}

// ---- unsorted event streams ---------------------------------------------------------------------------------------------------
// The reference loads the records into a std::multimap keyed by the time stamp (eventCameraCalib.cpp:154-163): any file order
// is accepted, equal stamps keep their file order.  The device equivalent: a stable radix sort of (stamp, index) and a gather.
namespace {
__global__ void k_ts_keys(const double *__restrict__ t, int64_t n, uint64_t *__restrict__ key, uint32_t *__restrict__ idx) {
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        key[i] = enc_d(t[i]);
        idx[i] = (uint32_t) i;
    }
}
__global__ void k_ts_gather(const uint32_t *__restrict__ idx, int64_t n, const double *__restrict__ t, const uint32_t *__restrict__ xyp,
                            double *__restrict__ t_out, uint32_t *__restrict__ xyp_out) {
    for (int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t) gridDim.x * blockDim.x) {
        const uint32_t o = idx[i];
        t_out[i] = t[o];
        xyp_out[i] = xyp[o];
    }
}
}  // namespace

int ecb_sort_events_by_time(ecb_ctx *ctx, int64_t n) {
    if (n <= 1) return ECB_OK;
    if (n >= 0xFFFFFFFFll) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "unsorted stream of %lld events", (long long) n);
    enum { B_KEY0 = 6, B_KEY1, B_IDX0, B_IDX1, B_HIST, B_T = 30, B_XYP = 31 };  // same slots as the general DBSCAN path
    DevBuf *B = ctx->gh;
    int rc;
    const size_t un = (size_t) n;
    const int nblk = (int) ((n + RS_TILE - 1) / RS_TILE);
    if ((rc = ecb_reserve(ctx, B[B_KEY0], un * 8))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_KEY1], un * 8))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_IDX0], un * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_IDX1], un * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_HIST], (size_t) 256 * nblk * 4))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_T], un * 8))) return rc;
    if ((rc = ecb_reserve(ctx, B[B_XYP], un * 4))) return rc;
    uint64_t *key[2] = {(uint64_t *) B[B_KEY0].p, (uint64_t *) B[B_KEY1].p};
    uint32_t *idx[2] = {(uint32_t *) B[B_IDX0].p, (uint32_t *) B[B_IDX1].p};
    const int g = grid_for(ctx, n);
    k_ts_keys<<<g, GH_THREADS, 0, ctx->stream>>>((const double *) ctx->ev_t.p, n, key[0], idx[0]);
    GH_LAUNCH(ctx, "k_ts_keys");
    int res = 0;
    if ((rc = gh_radix_sort(ctx, key, idx, n, 64, (uint32_t *) B[B_HIST].p, &res))) return rc;
    k_ts_gather<<<g, GH_THREADS, 0, ctx->stream>>>(idx[res], n, (const double *) ctx->ev_t.p, (const uint32_t *) ctx->ev_xyp.p,
                                                  (double *) B[B_T].p, (uint32_t *) B[B_XYP].p);
    GH_LAUNCH(ctx, "k_ts_gather");
    ECB_CUDA(ctx, cudaMemcpyAsync(ctx->ev_t.p, B[B_T].p, un * 8, cudaMemcpyDeviceToDevice, ctx->stream));
    ECB_CUDA(ctx, cudaMemcpyAsync(ctx->ev_xyp.p, B[B_XYP].p, un * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    return ECB_OK;
}
