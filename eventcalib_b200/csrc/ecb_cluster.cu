// k_cluster — the reference's DBSCAN (dbscan/include/dbscan.h:115-265 with the bundled kd-tree,
// dbscan/src/kdtree.cpp:106-179) for one point set per CTA, re-derived as data-parallel set operations on a
// shared-memory occupancy bitmap of the sensor plane (a perfect spatial hash with one pixel per cell):
//
//   1. occupancy bitmap U + word-prefix popcounts (pixel -> row-major rank)          [replaces the kd build]
//   2. level-synchronous emulation of the kd INSERTION ORDER (kd_insert in pid order, kdtree.cpp:106-146):
//      only two bits per point survive — "an ancestor splitting on axis d has the same d-coordinate" — which
//      is exactly when find_nearest (kdtree.cpp:166-171, `fabs(dx) < range`) misses a neighbour at q+eps*e_d
//   3. neighbour count = popcount of the eps-disc stencil on U, self excluded (dbscan.h:218), minus the
//      missed neighbours; core <=> count >= minPts (dbscan.h:151,247)
//   4. lock-free union-find over mutual core-core edges; the directed (one-way) edges left by the tie rule
//      are resolved by min-label propagation: cluster(G) = min seed pid over all groups that reach G
//      (equivalent to Run's ascending-pid seed loop + expandCluster BFS, dbscan.h:143-162,229-259)
//   5. cluster id = rank of the seed pid (discovery order); non-core points are Noise (dbscan.h:164-168)
//   6. cluster-size filter (CirclesEventFrame.cpp:89-117), member lists, exact integer moments for fitCircle
//      (CirclesEventFrame.cpp:364-404) and the median-by-norm member (CirclesEventFrame.cpp:137-147)
//
// HBM traffic per point: 4 B pixel read + 4 B label write + 4 B member write; everything else is on-chip.
#include <stdlib.h>

#include <algorithm>

#include "ecb_cluster.cuh"

namespace {

// RankT: rank of the first pixel of every pair of bitmap words (u16 while every problem has fewer than 65535 points).
// StT: r_st, per point the rank of a pid (steps 4 - 7), then the seed mask (8) and the member lists (9).  u16 (the narrow
// layout) needs pid < 2^15 and n <= KD_PT * threads: the slow kd path keeps its node pid and tie flags in one 32-bit word.
template <typename RankT, typename StT>
struct Smem {
    uint32_t *U, *C;
    RankT *wrank;
    uint32_t *r_pix, *r_lab, *r_kd;
    StT *r_st;
    uint8_t *r_flag;
};

// A/B switches of the round-2 changes (profiles/tools/ab_build.py builds variants with -D...=0)
// (warp-aggregated atomicMin in the first kd rounds was measured SLOWER: +0.18 ms on C2, MATCH.ANY costs more than the
// serialised atomics; profiles/r2d_ab_cluster.jsonl)
#ifndef ECB_CL_RANKORDER
#define ECB_CL_RANKORDER 1  // steps 5 - 6 walk the points in row-major rank order instead of pid order
#endif
#ifndef ECB_CL_ROLL
#define ECB_CL_ROLL 1     // one-or-two-trip bookkeeping loops stay rolled (code size)
#endif
#ifndef ECB_CL_UNSET
#define ECB_CL_UNSET 1      // planes cleared once per CTA, every problem un-sets the words it touched
#endif

constexpr int KD_PT = 6;  // points per thread kept in registers during the kd rounds (fast path: n <= KD_PT * threads)

__device__ __forceinline__ uint32_t find_root(volatile uint32_t *parent, uint32_t a) {
    uint32_t p = parent[a];
    while (p != a) {
        uint32_t g = parent[p];
        if (g != p) parent[a] = g;  // path halving (benign race: only ever points to an ancestor)
        a = p;
        p = g;
    }
    return a;
}

__device__ __forceinline__ void unite(uint32_t *parent, uint32_t a, uint32_t b) {
    for (;;) {
        a = find_root(parent, a);
        b = find_root(parent, b);
        if (a == b) return;
        if (a < b) {
            uint32_t t = a;
            a = b;
            b = t;
        }
        if (atomicCAS(&parent[a], a, b) == a) return;  // link the larger root under the smaller
    }
}

// SM = true: bit planes AND per-point arrays live in shared memory — every pointer below is then derived from the
// shared array alone, so the compiler emits LDS / STS / ATOMS with 32-bit addresses instead of generic accesses.
template <typename RankT, typename StT, bool SM>
__global__ void __launch_bounds__(ECB_CL_THREADS, 2) k_cluster(const ClusterArgs a) {
    extern __shared__ __align__(16) uint32_t smem_raw[];
    __shared__ uint32_t ws[33];
    __shared__ uint32_t s_nextpb[2], s_status, s_chunk;
    __shared__ uint8_t s_own[ECB_CL_THREADS / 32][32];  // 6b: lane of the k-th sub-run head of the warp's chunk

    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, wid = tid >> 5, nwarp = nthr >> 5;
    const int PW = a.PW, PH = a.PH, E = a.E, NW = PW * PH;
    const int NP = (NW + 1) >> 1;  // word pairs: one rank per pair (U is 8-byte aligned)
    Smem<RankT, StT> s;
    const int plane_words = 2 * NW + (int) ((NP * sizeof(RankT) + 3) / 4);
    uint32_t *arr;
    if constexpr (SM) {
        s.U = smem_raw;
        arr = smem_raw + plane_words;
    } else {
        uint32_t *gs = a.gscratch + (size_t) blockIdx.x * a.gscratch_stride;
        s.U = a.planes_in_smem ? smem_raw : gs;
        arr = a.planes_in_smem ? gs : gs + plane_words;
    }
    s.C = s.U + NW;
    s.wrank = reinterpret_cast<RankT *>(s.C + NW);
    const int NC = a.n_cap;
    s.r_pix = arr;
    s.r_lab = arr + NC;
    s.r_kd = arr + 2 * NC;  // 2*NC words
    const int st_words = sizeof(StT) == 4 ? NC : (NC + 1) >> 1;
    s.r_st = reinterpret_cast<StT *>(arr + 4 * NC);
    s.r_flag = reinterpret_cast<uint8_t *>(arr + (4 * NC + st_words));  // NC bytes, indexed by rank: kd tie flags (bit0 x, bit1 y)
    // kept-cluster scratch tables (raw id, size, member-list offset), max_k entries each (+1 for the end offset)
    int32_t *k_raw = reinterpret_cast<int32_t *>(arr + (4 * NC + st_words + ((NC + 3) >> 2)));
    int32_t *k_size = k_raw + a.max_k, *k_off = k_size + a.max_k;

    // ---- 0. clear planes: once per CTA; every problem un-sets the words it touched when it is done with them (step 8) ----
    for (int i = tid; i < 2 * NW; i += nthr) s.U[i] = 0;
    // Problems are drawn from a global counter.  The draw for the NEXT problem is issued at the start of the current one and
    // parked in a register of thread 0 until the header is written, so its latency (an L2 round trip per problem) is hidden.
    if (tid == 0) {
        s_nextpb[0] = atomicAdd(a.work_counter, 1u);
        s_status = 0;
    }
    for (int iter = 0;; ++iter) {
#if !ECB_CL_UNSET
        __syncthreads();
        for (int i = tid; i < 2 * NW; i += nthr) s.U[i] = 0;
#endif
        __syncthreads();
        const uint32_t pb = s_nextpb[iter & 1];
        if (pb >= (uint32_t) a.n_prob) break;
        uint32_t next_pb = 0;
        if (tid == 0) next_pb = atomicAdd(a.work_counter, 1u);
        const ProbDesc d = a.prob[pb];
        const int n = d.n;
        const uint32_t *gpix = a.pix[d.pol] + d.off;
        int32_t *glab = a.labels[d.pol] + d.off;
        // ---- 1. occupancy bitmap ---------------------------------------------------------------
        for (int pid = tid; pid < n; pid += nthr) {
            uint32_t p = gpix[pid];
            int x = (int) ECB_PIX_X(p) - d.x0, y = (int) ECB_PIX_Y(p) - d.y0;
            uint32_t loc = ECB_NONE;
            if (x >= 0 && x < a.W && y >= 0 && y < a.H && !(p & ECB_PIX_INVALID)) {
                x += E;
                y += E;
                uint32_t bit = 1u << (x & 31);
                uint32_t old = atomicOr(&s.U[y * PW + (x >> 5)], bit);
                if (old & bit)
                    atomicOr(&s_status, ECB_PB_DUPLICATE);
                else
                    loc = (uint32_t) x | ((uint32_t) y << 16);
            } else {
                atomicOr(&s_status, ECB_PB_RANGE);
            }
            s.r_pix[pid] = loc;
        }
        __syncthreads();
        // ---- 2. prefix popcounts per pair of words: rank(x,y) = wrank[pair] + popc(bits of the pair below) ----------
        // bits of pair i; an odd NW leaves the last pair with one word of U (the other is C[0])
        auto pair_bits = [&](int i) -> uint64_t { return 2 * i + 1 < NW ? reinterpret_cast<const uint64_t *>(s.U)[i] : (uint64_t) s.U[2 * i]; };
        uint32_t n_ranked;  // distinct in-range pixels = set bits of U (== n unless the input is flagged)
        {
            const int per = (NP + nthr - 1) / nthr;
            const int b = tid * per, e = min(NP, b + per);
            uint32_t c = 0;
#if ECB_CL_ROLL
#pragma unroll 1
#endif
            for (int i = b; i < e; ++i) c += __popcll(pair_bits(i));
            uint32_t ex = block_excl_scan(c, ws, &n_ranked);
#if ECB_CL_ROLL
#pragma unroll 1
#endif
            for (int i = b; i < e; ++i) {
                s.wrank[i] = (RankT) ex;
                ex += __popcll(pair_bits(i));
            }
        }
        __syncthreads();
        auto rank_of = [&](int x, int y) -> uint32_t {  // (x,y) occupied: only bits below it are counted
            const int w = y * PW + (x >> 5);
            const int b = ((w & 1) << 5) | (x & 31);
            return (uint32_t) s.wrank[w >> 1] + __popcll(reinterpret_cast<const uint64_t *>(s.U)[w >> 1] & ((1ull << b) - 1ull));
        };
        // ---- 4. kd insertion-order emulation -> tie flags ---------------------------------------
        // NOTE: the root is pid 0 like kd_insert's first insertion.
        uint32_t *child = s.r_kd;
        uint32_t *rloc = s.r_lab;  // [rank] -> packed pixel; r_lab is not needed before step 7
        for (int i = tid; i < 2 * n; i += nthr) child[i] = ECB_NONE;
        if (n <= KD_PT * nthr) {
            // fast path: each thread keeps its <= KD_PT points (pixel, current node, flags) in registers.
            // (Handing the last walkers of the late rounds over to one thread each was measured SLOWER: the rounds are bound by
            // the barrier + shared-memory latency chain, not by issue slots; profiles/r2s_ab_cluster_compact.jsonl.)
            uint32_t mypix[KD_PT], cur[KD_PT], fl[KD_PT];
#pragma unroll
            for (int k = 0; k < KD_PT; ++k) {
                const int pid = tid + k * nthr;
                mypix[k] = pid < n ? s.r_pix[pid] : ECB_NONE;
                cur[k] = (pid == 0 || mypix[k] == ECB_NONE) ? ECB_NONE : 0u;
                fl[k] = 0;
            }
            __syncthreads();
            for (int round = 0;; ++round) {
                const int dsh = (round & 1) ? 16 : 0;
                bool any = false;
                uint32_t slot[KD_PT];
#pragma unroll
                for (int k = 0; k < KD_PT; ++k) {
                    if (cur[k] == ECB_NONE) continue;
                    any = true;
                    const uint32_t ci = (mypix[k] >> dsh) & 0xFFFF, ca = (s.r_pix[cur[k]] >> dsh) & 0xFFFF;
                    if (ci == ca) fl[k] |= 1u << (round & 1);
                    slot[k] = 2 * cur[k] + (ci < ca ? 0 : 1);
                    atomicMin(&child[slot[k]], (uint32_t) (tid + k * nthr));
                }
                if (!__syncthreads_or(any)) break;
#pragma unroll
                for (int k = 0; k < KD_PT; ++k) {
                    if (cur[k] == ECB_NONE) continue;
                    const uint32_t c = child[slot[k]];
                    cur[k] = c == (uint32_t) (tid + k * nthr) ? ECB_NONE : c;
                }
                // no barrier needed here: a child slot is written only in the round in which its parent is reached,
                // and all points that reach a node do so in the same round
            }
#pragma unroll
            for (int k = 0; k < KD_PT; ++k)
                if (mypix[k] != ECB_NONE) {
                    const uint32_t rk = rank_of(mypix[k] & 0xFFFF, mypix[k] >> 16);
                    s.r_flag[rk] = (uint8_t) fl[k];
                    rloc[rk] = mypix[k];          // pixel of every rank: steps 5 - 6 walk the points in row-major order
                    s.r_st[tid + k * nthr] = (StT) rk;  // rank of every pid: step 7
                }
        } else if constexpr (sizeof(StT) == 4) {  // the launcher picks the narrow layout only where the fast path runs
            uint32_t *state = s.r_st;
            const uint32_t DONE = 0x3FFFFFFFu;
            for (int pid = tid; pid < n; pid += nthr) state[pid] = (pid == 0 || s.r_pix[pid] == ECB_NONE) ? DONE : 0u;
            __syncthreads();
            for (int round = 0;; ++round) {
                const int dsh = (round & 1) ? 16 : 0;
                bool any = false;
                for (int pid = tid; pid < n; pid += nthr) {
                    uint32_t st = state[pid];
                    uint32_t cur = st & DONE;
                    if (cur == DONE) continue;
                    any = true;
                    uint32_t ci = (s.r_pix[pid] >> dsh) & 0xFFFF, ca = (s.r_pix[cur] >> dsh) & 0xFFFF;
                    if (ci == ca) state[pid] = st | (0x40000000u << (round & 1));
                    atomicMin(&child[2 * cur + (ci < ca ? 0 : 1)], (uint32_t) pid);
                }
                if (!__syncthreads_or(any)) break;
                for (int pid = tid; pid < n; pid += nthr) {
                    uint32_t st = state[pid];
                    uint32_t cur = st & DONE;
                    if (cur == DONE) continue;
                    uint32_t ci = (s.r_pix[pid] >> dsh) & 0xFFFF, ca = (s.r_pix[cur] >> dsh) & 0xFFFF;
                    uint32_t c = child[2 * cur + (ci < ca ? 0 : 1)];
                    state[pid] = (st & 0xC0000000u) | (c == (uint32_t) pid ? DONE : c);
                }
                __syncthreads();
            }
            for (int pid = tid; pid < n; pid += nthr) {
                const uint32_t loc = s.r_pix[pid];
                if (loc != ECB_NONE) {
                    const uint32_t rk = rank_of(loc & 0xFFFF, loc >> 16);
                    s.r_flag[rk] = (uint8_t) (state[pid] >> 30);
                    rloc[rk] = loc;
                    state[pid] = rk;  // r_st: same thread, same index as the read above
                }
            }
        }
        __syncthreads();
        if (a.exact_order) {  // the emulated tree itself, for the member-order pass: one 16-byte node per point
            uint32_t *nodes = a.kd_nodes[d.pol] + 4 * d.off;  // {pixel, left, right, parent}
            for (int pid = tid; pid < n; pid += nthr) {
                const uint32_t l = child[2 * pid], r = child[2 * pid + 1];
                nodes[4 * pid] = gpix[pid];
                nodes[4 * pid + 1] = l;
                nodes[4 * pid + 2] = r;
                if (l != ECB_NONE) nodes[4 * l + 3] = (uint32_t) pid;
                if (r != ECB_NONE) nodes[4 * r + 3] = (uint32_t) pid;
            }
            if (tid == 0 && n > 0) nodes[3] = ECB_NONE;
            __syncthreads();  // `child` (r_kd) is re-used as parent / glabel below
        }
        // tie flag of the (occupied) pixel (x,y): bit0 = FX, bit1 = FY
        auto flag_of = [&](int x, int y) -> uint32_t { return s.r_flag[rank_of(x, y)]; };
        // ---- 5. neighbour count, core flag -----------------------------------------------------------
        // (steps 5, 6a, 6b take the points in row-major RANK order: neighbouring lanes then read the same or adjacent bitmap
        // words — broadcasts instead of the bank conflicts of the pid order, which is the hash-set order, i.e. random)
        const int ei = a.eps_int;
        const int m = (int) n_ranked;
        for (int it5 = tid; it5 < (ECB_CL_RANKORDER ? m : n); it5 += nthr) {
            int rk = it5;
            if (!ECB_CL_RANKORDER) {
                if (s.r_pix[it5] == ECB_NONE) continue;
                rk = (int) s.r_st[it5];
            }
            const uint32_t loc = rloc[rk];
            const int x = loc & 0xFFFF, y = loc >> 16;
            int cnt = -1;  // self
            for (int dy = -E; dy <= E; ++dy) {
                const int w = a.halfw[dy < 0 ? -dy : dy];
                cnt += __popc(row_bits(s.U + (y + dy) * PW, x - w, 2 * w + 1));
            }
            if (ei > 0) {  // neighbours the kd query misses (kdtree.cpp:166-171)
                if (test_bit(s.U + y * PW, x + ei)) cnt -= (int) (flag_of(x + ei, y) & 1u);
                if (test_bit(s.U + (y + ei) * PW, x)) cnt -= (int) ((flag_of(x, y + ei) >> 1) & 1u);
            }
            if (cnt >= (int) a.min_pts) atomicOr(&s.C[y * PW + (x >> 5)], 1u << (x & 31));
        }
        uint32_t *parent = s.r_kd, *glabel = s.r_kd + NC;
        for (int r = tid; r < n; r += nthr) {
            parent[r] = r;
            glabel[r] = ECB_NONE;
        }
        __syncthreads();
        // ---- 6. connected components over mutual core edges ---------------------------------------------
        // Inside one bitmap row, core pixels less than eps apart are always mutually adjacent (the tie rule only concerns
        // distance exactly eps).  6a: every core pixel points straight at the first pixel of its in-row run (gaps <= gap),
        // found with bit scans — no atomics, depth-1 trees.  6b/6c: runs are then united across rows (and across an
        // exact-eps in-row gap) with a lock-free union-find whose chains start at run heads.
        const int gap = (ei > 0 ? ei : E + 1) - 1;  // pixels whose distance is <= gap are unconditionally adjacent in-row
        for (int it6 = tid; it6 < (ECB_CL_RANKORDER ? m : n); it6 += nthr) {
            int rk = it6;
            if (!ECB_CL_RANKORDER) {
                if (s.r_pix[it6] == ECB_NONE) continue;
                rk = (int) s.r_st[it6];
            }
            const uint32_t loc = rloc[rk];
            const int x = loc & 0xFFFF, y = loc >> 16;
            if (!test_bit(s.C + y * PW, x)) continue;
            int p = x;
            if (gap > 0)
                for (;;) {  // hop to the farthest core pixel within `gap` to the left until there is none
                    const uint32_t wbits = row_bits(s.C + y * PW, p - gap, gap);
                    if (!wbits) break;
                    p = p - gap + (__ffs(wbits) - 1);
                }
            if (p != x) parent[rk] = rank_of(p, y);
        }
        if (tid == 0) s_chunk = 0;
        __syncthreads();
        // 6b/6c work item = core pixel.  Every pixel tests its exact-eps in-row link (dy = 0); the inter-row unions are done
        // by the FIRST pixel of every sub-run of its bitmap word only (sub-run = core pixels of the word with gaps <= gap),
        // so an adjacent (sub-run, run) pair is united once instead of once per pixel pair: the sub-run is dilated by the
        // half width of the eps-disc at dy and intersected with row y + dy, and the first pixel of every run in the
        // intersection is united with the sub-run's first pixel.  dy = eps (half width 0): pixel pairs in the same column,
        // minus the ones the kd query misses (one-way edges, see 7).
        {
            auto smear = [&](uint64_t v) -> uint64_t {  // OR of (v << 1 .. v << gap)
                uint64_t sm = v;
                for (int k = 0; k < gap - 1;) {
                    const int add = min(k + 1, gap - 1 - k);
                    sm |= sm << add;
                    k += add;
                }
                return gap > 0 ? sm << 1 : 0ull;
            };
            // Load balance: warps draw chunks of 32 ranks from a shared counter, and inside a warp the (sub-run head, dy) pairs
            // of the chunk are dealt out evenly to the lanes (the union cost per pair varies a lot).
            const uint32_t invE = (65536u + (uint32_t) E - 1u) / (uint32_t) E;  // it / E == (it * invE) >> 16 for it < 512
            for (;;) {
                int base = 0;
                if (lane == 0) base = (int) atomicAdd(&s_chunk, 32u);
                base = __shfl_sync(0xffffffffu, base, 0);
                if (base >= (ECB_CL_RANKORDER ? m : n)) break;
                int rk = base + lane;
                bool head = false;
                uint32_t h_xy = 0, h_sub = 0, h_rf = 0;
                bool have = rk < m;
                if (!ECB_CL_RANKORDER) {
                    have = rk < n && s.r_pix[rk] != ECB_NONE;
                    if (have) rk = (int) s.r_st[rk];
                }
                if (have) {
                    const uint32_t loc = rloc[rk];
                    {
                        const int x = loc & 0xFFFF, y = loc >> 16;
                        const int j = x >> 5, f = x & 31;
                        const uint32_t *crow = s.C + y * PW;
                        const uint32_t src = crow[j];
                        if ((src >> f) & 1u) {
                            // q = p - eps*e_x with nothing in between: mutual unless the kd query misses q -> p (FX(p))
                            if (ei > 0 && test_bit(crow, x + ei) && !row_bits(crow, x + 1, ei - 1) &&
                                !(flag_of(x + ei, y) & 1u))
                                unite(parent, (uint32_t) rk, rank_of(x + ei, y));
                            const uint32_t F = src & ~(uint32_t) smear(src);  // first pixel of every sub-run of the word
                            if ((F >> f) & 1u) {
                                const uint32_t Fup = f < 31 ? F >> (f + 1) : 0u;  // next sub-run start above f
                                const uint32_t upto = Fup ? ((1u << (f + __ffs(Fup))) - 1u) : 0xFFFFFFFFu;
                                head = true;
                                h_xy = loc;
                                h_sub = src & upto & ~((1u << f) - 1u);
                                h_rf = (uint32_t) rk;
                            }
                        }
                    }
                }
                const uint32_t hm = __ballot_sync(0xffffffffu, head);
                if (head) s_own[wid][__popc(hm & ((1u << lane) - 1u))] = (uint8_t) lane;
                __syncwarp();
                const int n_it = __popc(hm) * E;
                for (int it0 = 0; it0 < n_it; it0 += 32) {
                    const int it = it0 + lane;
                    const bool act = it < n_it;
                    const int hi = act ? (int) (((uint32_t) it * invE) >> 16) : 0;
                    const int dy = it - hi * E + 1;
                    const int owner = (int) s_own[wid][hi];
                    const uint32_t loc = __shfl_sync(0xffffffffu, h_xy, owner);
                    const uint32_t sub = __shfl_sync(0xffffffffu, h_sub, owner);
                    const uint32_t rf = __shfl_sync(0xffffffffu, h_rf, owner);
                    if (!act) continue;
                    const int x = loc & 0xFFFF, y = loc >> 16, j = x >> 5;
                    const int w = a.halfw[dy];
                    const uint32_t *tr = s.C + (y + dy) * PW + j;  // word j of row y + dy
                    const uint32_t T0 = j > 0 ? tr[-1] : 0u, T1 = tr[0], T2 = j + 1 < PW ? tr[1] : 0u;
                    if (!(T0 | T1 | T2)) continue;
                    const uint64_t Tw = ((uint64_t) T0 >> 16) | ((uint64_t) T1 << 16) | ((uint64_t) T2 << 48);  // bit k = pixel 32j-16+k
                    uint64_t d64 = ((uint64_t) sub << 16) >> w;  // bits >= 16 - w >= 1
                    for (int k = 0; k < 2 * w;) {  // OR of shifts 0..2w: the sub-run dilated by w (top bit <= 47 + w)
                        const int add = min(k + 1, 2 * w - k);
                        d64 |= d64 << add;
                        k += add;
                    }
                    uint64_t hits = d64 & Tw;
                    if (!hits) continue;
                    if (dy != ei) hits &= ~smear(hits);  // first pixel of every run of the intersection
                    while (hits) {
                        const int nx = 32 * j - 16 + (__ffsll((long long) hits) - 1);
                        hits &= hits - 1;
                        // dy = eps: q -> p missed by the kd query: the pair is a one-way edge p -> q (handled in 7)
                        if (dy == ei && (flag_of(nx, y + dy) & 2u)) continue;
                        unite(parent, rf, rank_of(nx, y + dy));
                    }
                }
                __syncwarp();  // s_own is rewritten by the next chunk
            }
        }
        __syncthreads();
        // ---- 7. flatten, group min pid, one-way edge propagation --------------------------------------
        int n_core_local = 0;
        for (int pid = tid; pid < n; pid += nthr) {
            uint32_t loc = s.r_pix[pid];
            uint32_t root = ECB_NONE;
            if (loc != ECB_NONE) {
                const int x = loc & 0xFFFF, y = loc >> 16;
                if (test_bit(s.C + y * PW, x)) {
                    ++n_core_local;
                    root = find_root(parent, s.r_st[pid]);
                    atomicMin(&glabel[root], (uint32_t) pid);
                }
            }
            s.r_lab[pid] = root;  // stash: root rank of the point's group (ECB_NONE for non-core); rloc is dead since 6b's barrier
        }
        __syncthreads();
        for (int pid = tid; pid < n; pid += nthr) {  // full flatten: parent[rank] = root for every core point
            const uint32_t root = s.r_lab[pid];
            if (root != ECB_NONE) parent[s.r_st[pid]] = root;
        }
        __syncthreads();
        if (ei > 0) {
            for (;;) {
                bool changed = false;
                for (int pid = tid; pid < n; pid += nthr) {
                    const uint32_t gq = s.r_lab[pid];
                    if (gq == ECB_NONE) continue;
                    const uint32_t loc = s.r_pix[pid];
                    const int x = loc & 0xFFFF, y = loc >> 16;
                    // p = q + eps*e_x with FX(p): edge p -> q only
                    if (test_bit(s.C + y * PW, x + ei)) {
                        const uint32_t rp = rank_of(x + ei, y);
                        if (s.r_flag[rp] & 1u) {
                            uint32_t lp = ((volatile uint32_t *) glabel)[parent[rp]];
                            if (lp < atomicMin(&glabel[gq], lp)) changed = true;
                        }
                    }
                    if (test_bit(s.C + (y + ei) * PW, x)) {
                        const uint32_t rp = rank_of(x, y + ei);
                        if (s.r_flag[rp] & 2u) {
                            uint32_t lp = ((volatile uint32_t *) glabel)[parent[rp]];
                            if (lp < atomicMin(&glabel[gq], lp)) changed = true;
                        }
                    }
                }
                if (!__syncthreads_or(changed)) break;
            }
        }
        // ---- 8. seeds -> cluster ids ---------------------------------------------------------------------
        const int nw32 = (n + 31) >> 5;
        uint32_t *seedmask = reinterpret_cast<uint32_t *>(s.r_st), *seedpref = seedmask + nw32;  // 8 * nw32 <= NC * sizeof(StT) bytes
        for (int i = tid; i < nw32; i += nthr) seedmask[i] = 0;
        __syncthreads();
        for (int pid = tid; pid < n; pid += nthr) {
            const uint32_t g = s.r_lab[pid];
            if (g == ECB_NONE) continue;
            // a group is a seed iff its final label is one of its own members (nothing smaller reached it);
            // the member with pid == glabel[g] marks it
            if (glabel[g] == (uint32_t) pid) atomicOr(&seedmask[pid >> 5], 1u << (pid & 31));
        }
        __syncthreads();
        uint32_t n_clusters;
        {
            const int per = (nw32 + nthr - 1) / nthr;
            const int b = tid * per, e = min(nw32, b + per);
            uint32_t c = 0;
#if ECB_CL_ROLL
#pragma unroll 1
#endif
            for (int i = b; i < e; ++i) c += __popc(seedmask[i]);
            uint32_t ex = block_excl_scan(c, ws, &n_clusters);
#if ECB_CL_ROLL
#pragma unroll 1
#endif
            for (int i = b; i < e; ++i) {
                seedpref[i] = ex;
                ex += __popc(seedmask[i]);
            }
        }
        __syncthreads();
        for (int pid = tid; pid < n; pid += nthr) {
            const uint32_t g = s.r_lab[pid];
            int32_t lab = -1;
            if (g != ECB_NONE) {
                const uint32_t seed = glabel[g];
                lab = (int32_t) (seedpref[seed >> 5] + __popc(seedmask[seed >> 5] & ((1u << (seed & 31)) - 1u)));
            }
            s.r_lab[pid] = (uint32_t) lab;
            glab[pid] = lab;
            const uint32_t loc = s.r_pix[pid];  // U and C are dead: leave the planes empty for the CTA's next problem
            if (ECB_CL_UNSET && loc != ECB_NONE) {
                const int w = (int) (loc >> 16) * PW + (int) ((loc & 0xFFFF) >> 5);
                s.U[w] = 0;
                s.C[w] = 0;
            }
        }
        __syncthreads();
        // ---- 9. cluster sizes, size filter, member lists, moments, medians ----------------------------
        const int nc = (int) n_clusters;
        uint32_t *csize = s.r_kd, *keptidx = s.r_kd + nc;  // nc <= n <= NC; the rest of r_kd is scratch
        for (int i = tid; i < nc; i += nthr) csize[i] = 0;
        __syncthreads();
        for (int pid = tid; pid < n; pid += nthr) {
            int32_t lab = (int32_t) s.r_lab[pid];
            if (lab >= 0) atomicAdd(&csize[lab], 1u);
        }
        __syncthreads();
        uint32_t n_kept = 0;
        {
            const int per = (nc + nthr - 1) / nthr;
            const int b = tid * per, e = min(nc, b + per);
            uint32_t c = 0;
#if ECB_CL_ROLL
#pragma unroll 1
#endif
            for (int i = b; i < e; ++i) c += csize[i] >= a.cluster_min;
            uint32_t ex = block_excl_scan(c, ws, &n_kept);
#if ECB_CL_ROLL
#pragma unroll 1
#endif
            for (int i = b; i < e; ++i) {
                const bool k = csize[i] >= a.cluster_min;
                keptidx[i] = k ? ex : ECB_NONE;
                if (k && ex < (uint32_t) a.max_k) {
                    k_raw[ex] = i;
                    k_size[ex] = (int32_t) csize[i];
                }
                ex += k;
            }
        }
        if (n_kept > (uint32_t) a.max_k) {
            if (tid == 0) {
                atomicOr(&s_status, ECB_PB_CLUSTER_CAP);
                if (a.max_kept) atomicMax(a.max_kept, n_kept);  // the caller re-runs with a table of that capacity
            }
            n_kept = a.max_k;
        }
        __syncthreads();
        if (wid == 0) {  // member-list offsets: exclusive scan of k_size[0..n_kept)
            uint32_t run = 0;
#if ECB_CL_ROLL
#pragma unroll 1
#endif
            for (int base = 0; base < (int) n_kept; base += 32) {
                uint32_t v = base + lane < (int) n_kept ? (uint32_t) k_size[base + lane] : 0;
                uint32_t inc = warp_incl_scan(v);
                if (base + lane < (int) n_kept) k_off[base + lane] = (int32_t) (run + inc - v);
                run += __shfl_sync(0xffffffffu, inc, 31);
            }
            if (lane == 0) k_off[n_kept] = (int32_t) run;
        }
        __syncthreads();
        StT *members = s.r_st;  // seedmask/seedpref are dead
        uint32_t *gmem = a.kmem[d.pol] + d.off;
        KeptCluster *kt = a.ktab + (size_t) pb * a.max_k;
        if (n_kept > 0) {
            // Ordered member lists (ascending pid inside every cluster) without scanning all points once per cluster:
            // each warp owns a contiguous pid range; pass A counts its members per kept cluster, a scan over the warps
            // turns the counts into start positions, pass B places.  Counters live in the free tail of r_kd.
            const int L = (((n + nwarp - 1) / nwarp) + 31) & ~31;  // pids per warp, multiple of 32
            const int p0 = wid * L, p1 = min(n, p0 + L);
            auto kept_of = [&](int pid) -> int {
                if (pid >= p1) return -1;
                const int32_t lab = (int32_t) s.r_lab[pid];
                if (lab < 0) return -1;
                const uint32_t ki = keptidx[lab];
                return (ki != ECB_NONE && ki < n_kept) ? (int) ki : -1;
            };
            if ((int) n_kept * nwarp <= 2 * NC - 2 * nc) {
                uint32_t *cnt = s.r_kd + 2 * nc;
                for (int i = tid; i < (int) n_kept * nwarp; i += nthr) cnt[i] = 0;
                __syncthreads();
                uint32_t *mycnt = cnt + wid * n_kept;
                for (int c = p0; c < p1; c += 32) {
                    const int kidx = kept_of(c + lane);
                    const uint32_t peers = __match_any_sync(0xffffffffu, kidx);
                    if (kidx >= 0 && (peers & ((1u << lane) - 1u)) == 0) mycnt[kidx] += __popc(peers);
                    __syncwarp();
                }
                __syncthreads();
#if ECB_CL_ROLL
#pragma unroll 1
#endif
                for (int k = tid; k < (int) n_kept; k += nthr) {
                    uint32_t run = 0;
#if ECB_CL_ROLL
#pragma unroll 1
#endif
                    for (int w = 0; w < nwarp; ++w) {
                        const uint32_t t = cnt[w * n_kept + k];
                        cnt[w * n_kept + k] = run;
                        run += t;
                    }
                }
                __syncthreads();
                for (int c = p0; c < p1; c += 32) {
                    const int pid = c + lane;
                    const int kidx = kept_of(pid);
                    const uint32_t peers = __match_any_sync(0xffffffffu, kidx);
                    const int rk = __popc(peers & ((1u << lane) - 1u));
                    uint32_t base = 0;
                    if (kidx >= 0) {
                        base = mycnt[kidx];
                        members[k_off[kidx] + base + rk] = (StT) pid;
                    }
                    __syncwarp();
                    if (kidx >= 0 && rk == 0) mycnt[kidx] = base + __popc(peers);
                    __syncwarp();
                }
            } else {
                // many kept clusters: one warp per cluster scans the labels (O(n_kept * n / 32))
                for (int k = wid; k < (int) n_kept; k += nwarp) {
                    const int32_t cid = k_raw[k];
                    const int base = k_off[k];
                    int pos = 0;
                    for (int st = 0; st < n; st += 32) {
                        const int pid = st + lane;
                        const bool m = pid < n && (int32_t) s.r_lab[pid] == cid;
                        const uint32_t ball = __ballot_sync(0xffffffffu, m);
                        if (m) members[base + pos + __popc(ball & ((1u << lane) - 1u))] = (StT) pid;
                        pos += __popc(ball);
                    }
                }
            }
        }
        __syncthreads();
        // median keys fit one word when norm^2 * 2^bits(pid) < 2^32 (DAVIS346: 18 + 12 bits)
        const int pbits = 32 - __clz(max(n - 1, 1));
        const unsigned long long maxn2 = (unsigned long long) (a.W - 1 + d.x0) * (a.W - 1 + d.x0) +
                                         (unsigned long long) (a.H - 1 + d.y0) * (a.H - 1 + d.y0);
        const bool key32 = pbits < 32 && maxn2 < (1ull << (32 - pbits));
        for (int k = wid; k < (int) n_kept; k += nwarp) {
            const int32_t cid = k_raw[k];
            const int base = k_off[k], sz = k_size[k];
            // pixel coordinates are in [0, 32767]: squares and x*y are exact in 32 bits, cubes are one 32 x 32 -> 64 multiply-add
            unsigned long long S[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
            int med = -1;
            uint32_t *mnorm = s.r_kd;  // csize / keptidx are dead: squared norms of the members, same indexing as `members`
            for (int i = lane; i < sz; i += 32) {
                const uint32_t pid = members[base + i];
                gmem[base + i] = pid;
                const uint32_t loc = s.r_pix[pid];
                const uint32_t x = (uint32_t) ((int) (loc & 0xFFFF) - E + d.x0), y = (uint32_t) ((int) (loc >> 16) - E + d.y0);
                const uint32_t xx = x * x, yy = y * y, xy = x * y;
                S[0] += x;
                S[1] += y;
                S[2] += xx;
                S[3] += yy;
                S[4] += xy;
                S[5] += (unsigned long long) xx * x;
                S[6] += (unsigned long long) yy * y;
                S[7] += (unsigned long long) xy * y;
                S[8] += (unsigned long long) xx * y;
                mnorm[base + i] = xx + yy;
            }
            __syncwarp();
            bool tie = false;
            if (key32) {
                // (norm^2, pid) packed into one word: one shared load and one compare per pair
#if ECB_CL_ROLL
#pragma unroll 1
#endif
                for (int i = lane; i < sz; i += 32) mnorm[base + i] = (mnorm[base + i] << pbits) | members[base + i];
                __syncwarp();
                uint32_t mkey = 0;
                for (int i = lane; i < sz; i += 32) {  // rank among the members; slot sz/2 is the median
                    const uint32_t ki = mnorm[base + i];
                    int cnt = 0;
                    for (int j = 0; j < sz; ++j) cnt += mnorm[base + j] < ki;
                    if (cnt == sz / 2) mkey = ki;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mkey = max(mkey, __shfl_xor_sync(0xffffffffu, mkey, o));
                med = (int) (mkey & ((1u << pbits) - 1u));
                int eq = 0;  // std::nth_element's pick among equal norms depends on the member order
#if ECB_CL_ROLL
#pragma unroll 1
#endif
                for (int i = lane; i < sz; i += 32) eq += (mnorm[base + i] >> pbits) == (mkey >> pbits);
                tie = __reduce_add_sync(0xffffffffu, eq) > 1;
                if (lane != 0) med = -1;
            } else {
                for (int i = lane; i < sz; i += 32) {  // rank of (norm^2, pid) among the members; slot sz/2 is the median
                    const uint32_t ni = mnorm[base + i], pi = members[base + i];
                    int cnt = 0, eq = 0;
                    for (int j = 0; j < sz; ++j) {
                        const uint32_t nj = mnorm[base + j], pj = members[base + j];
                        cnt += (nj < ni) || (nj == ni && pj < pi);
                        eq += nj == ni;
                    }
                    if (cnt == sz / 2) {
                        med = (int) pi;
                        tie = eq > 1;
                    }
                }
            }
            if (a.exact_order && __any_sync(0xffffffffu, tie) && lane == 0) {
                const unsigned slot = atomicAdd(a.bfs_count, 1u);
                if (slot < (unsigned) a.bfs_cap) {
                    BfsItem it;
                    it.pb = (int32_t) pb;
                    it.cid = cid;
                    it.seed = (int32_t) members[base];  // ascending pid list: the seed is its first entry
                    it.size = sz;
                    it.mem_off = base;
                    it.kept = k;
                    a.bfs_items[slot] = it;
                }
            }
            // warp sums with the integer reduction unit: three 21-bit limbs per 64-bit partial sum (each < 2^63)
#pragma unroll
            for (int q = 0; q < 9; ++q) {
                const uint32_t l0 = __reduce_add_sync(0xffffffffu, (uint32_t) S[q] & 0x1FFFFFu);
                const uint32_t l1 = __reduce_add_sync(0xffffffffu, (uint32_t) (S[q] >> 21) & 0x1FFFFFu);
                const uint32_t l2 = __reduce_add_sync(0xffffffffu, (uint32_t) (S[q] >> 42));
                S[q] = (unsigned long long) l0 + ((unsigned long long) l1 << 21) + ((unsigned long long) l2 << 42);
            }
            med = __reduce_max_sync(0xffffffffu, med);
            if (lane == 0) {
                KeptCluster kc;
                kc.raw_id = cid;
                kc.size = sz;
                kc.med_pid = med;
                const uint32_t lm = s.r_pix[med];
                kc.med_x = (int) (lm & 0xFFFF) - E + d.x0;
                kc.med_y = (int) (lm >> 16) - E + d.y0;
                kc.mem_off = base;
#pragma unroll
                for (int q = 0; q < 9; ++q) kc.m[q] = (double) S[q];
                kt[k] = kc;
            }
        }
        // ---- header -------------------------------------------------------------------------------------
        {
            uint32_t tot;
            block_excl_scan((uint32_t) n_core_local, ws, &tot);
            if (tid == 0) {
                ProbHdr h;
                h.n_clusters = nc;
                h.n_kept = (int32_t) n_kept;
                h.n_core = (int32_t) tot;
                h.status = s_status;
                a.hdr[pb] = h;
                s_status = 0;
                s_nextpb[(iter + 1) & 1] = next_pb;
            }
        }
    }
}

}  // namespace

// words of the per-point arrays + the kept-cluster scratch tables of one CTA (st16: r_st as 16-bit words)
static size_t cluster_array_words(int n_cap, int max_k, bool st16) {
    return (size_t) 4 * n_cap + (st16 ? ((size_t) n_cap + 1) / 2 : (size_t) n_cap) + ((size_t) n_cap + 3) / 4 +
           (size_t) 3 * max_k + 1;
}

size_t ecb_cluster_smem_bytes(int PW, int PH, int n_cap, int max_k, bool arrays_in_smem, bool rank32, bool st16) {
    size_t NP = ((size_t) PW * PH + 1) / 2;
    size_t b = (size_t) PW * PH * 8 + ((NP * (rank32 ? 4 : 2) + 3) / 4) * 4;
    if (arrays_in_smem) b += cluster_array_words(n_cap, max_k, st16) * 4;
    return b;
}

int ecb_launch_cluster(ecb_ctx *ctx, ClusterArgs &a, int max_n) {
    if (a.n_prob <= 0) return ECB_OK;
    const bool rank32 = max_n >= 65535;
    a.n_cap = max_n < 64 ? 64 : max_n;
    // static shared + reserve; also the (constant) dynamic-smem attribute value, so that concurrent launches from several
    // host threads with different sizes cannot race on cudaFuncSetAttribute
    const size_t limit = (size_t) ctx->smem_optin - 9 * 1024;
    const size_t planes = ecb_cluster_smem_bytes(a.PW, a.PH, a.n_cap, a.max_k, false, rank32, false);
    // sensors whose bit planes exceed one CTA's shared memory (e.g. 1280x720) run with the planes in per-CTA L2 scratch
    a.planes_in_smem = planes <= limit;
    // CTA size: the kernel is barrier / latency bound, so more independent CTAs per SM beat bigger ones.  Shared memory
    // decides how many CTAs fit (DAVIS346 at 1 235 points per problem: 54 KB -> 4); at 64 registers an SM holds 1024
    // threads, so each CTA gets 1024 / CTAs threads (3 CTAs x 320 threads measured 16 % faster than 2 x 512).
    // The narrow layout (16-bit r_st) is taken wherever it can run: pid < 2^15 and the fast kd path covers the batch.
    void (*kern)(const ClusterArgs) = nullptr;
    size_t smem = 0;
    int threads = ECB_CL_THREADS;
    for (int st16 = a.n_cap < 32768; st16 >= 0; --st16) {
        const size_t with_arrays = ecb_cluster_smem_bytes(a.PW, a.PH, a.n_cap, a.max_k, true, rank32, st16);
        a.arrays_in_smem = with_arrays <= limit;  // else the per-point arrays live in per-CTA L2 scratch
        if (st16 && !a.arrays_in_smem) continue;
        smem = a.arrays_in_smem ? with_arrays : (a.planes_in_smem ? planes : 0);
        kern = st16 ? k_cluster<uint16_t, uint16_t, true>
             : rank32 ? (a.arrays_in_smem ? k_cluster<uint32_t, uint32_t, true> : k_cluster<uint32_t, uint32_t, false>)
                      : (a.arrays_in_smem ? k_cluster<uint16_t, uint32_t, true> : k_cluster<uint16_t, uint32_t, false>);
        ECB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) limit));
        int by_smem = 1;
        ECB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&by_smem, kern, 32, smem));
        threads = std::max(128, std::min(ECB_CL_THREADS, (1024 / std::max(by_smem, 1)) & ~31));
        if (!a.arrays_in_smem) threads = ECB_CL_THREADS;  // large problems in L2 scratch: few CTAs, each wants all the threads it can get
        if (const char *e = getenv("ECB_CL_THREADS")) threads = std::max(64, std::min(ECB_CL_THREADS, atoi(e) & ~31));
        if (!st16 || a.n_cap <= KD_PT * threads) break;
    }
    int per_sm = 1;
    ECB_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
    if (per_sm < 1) per_sm = 1;
    int grid = ctx->sm_count * per_sm;
    if (grid > a.n_prob) grid = a.n_prob;
    if (!a.arrays_in_smem) {
        // even: the bit planes at the start of a CTA's slice are read as 64-bit word pairs
        a.gscratch_stride = (cluster_array_words(a.n_cap, a.max_k, false) + (a.planes_in_smem ? 0 : (planes + 3) / 4) + 1) & ~(size_t) 1;
        int rc = ecb_reserve(ctx, ctx->scratch, (size_t) grid * a.gscratch_stride * 4);
        if (rc) return rc;
        a.gscratch = (uint32_t *) ctx->scratch.p;
    }
    ECB_CUDA(ctx, cudaMemsetAsync(a.work_counter, 0, 4, ctx->stream));
    ECB_PROF_BEGIN(ctx, ECB_STAGE_CLUSTER);
    kern<<<grid, threads, smem, ctx->stream>>>(a);
    ECB_PROF_END(ctx, ECB_STAGE_CLUSTER);
    ECB_LAUNCHED(ctx);
    return ecb_check(ctx, cudaGetLastError(), "k_cluster launch");
}
