// Device-side structures shared by the window, cluster and pair kernels.
#pragma once
#include "ecb_common.cuh"

#define ECB_CL_THREADS 512

// one clustering problem = one (window, polarity) point set, or one ecb_dbscan_run input
struct ProbDesc {
    int64_t off;      // offset of the problem's points in pix[pol] / labels[pol] / kmem[pol]
    int32_t n;        // number of points (pid = 0..n-1)
    int32_t pol;      // which flat array
    int32_t x0, y0;   // origin subtracted before indexing the bitmap
    int32_t pad0, pad1;
};

struct ProbHdr {
    int32_t n_clusters;  // raw clusters (discovery order ids 0..n_clusters-1)
    int32_t n_kept;      // clusters with size >= cluster_min (clipped to max_k)
    int32_t n_core;
    uint32_t status;     // ECB_PB_*
};

struct KeptCluster {
    int32_t raw_id;
    int32_t size;
    int32_t med_pid;   // member with the median norm (slot size/2 of the members sorted by (norm^2, pid))
    int32_t med_x, med_y;
    int32_t mem_off;   // offset of the member list inside the problem's kmem slice
    double m[9];       // Sx Sy Sxx Syy Sxy Sxxx Syyy Sxyy Sxxy (exact integers)
};

// one cluster whose members must be put in the reference's BFS pop order (k_bfs_order, ecb_bfs.cu)
struct BfsItem {
    int32_t pb;        // problem
    int32_t cid;       // raw cluster id (label)
    int32_t seed;      // lowest pid of the cluster = the point Run() started it from
    int32_t size;
    int32_t mem_off;   // offset of the member list inside the problem's member slice
    int32_t kept;      // index into the problem's KeptCluster table whose median is to be re-selected, or -1
};

struct ClusterArgs {
    const ProbDesc *prob;
    int n_prob;
    unsigned *work_counter;
    const uint32_t *pix[2];
    int32_t *labels[2];
    uint32_t *kmem[2];
    ProbHdr *hdr;
    KeptCluster *ktab;
    int max_k;
    uint32_t *max_kept;         // device word (may be null): atomicMax of the kept-cluster count of problems that overflow max_k
    uint32_t *gscratch;         // per-CTA global scratch when the per-point arrays do not fit shared memory
    size_t gscratch_stride;     // words per CTA
    int arrays_in_smem;
    int planes_in_smem;         // 0: sensor too large for one CTA's shared memory, the bit planes live in the L2 scratch too
    int n_cap;                  // region size (>= max n over the batch, >= 64)
    int W, H, E, PW, PH;        // bitmap: W x H pixels, E = floor(eps) padding, PW words per padded row, PH rows
    int eps_int;                // eps if it is an integer (the kd tie rule can fire), else -1
    uint32_t min_pts, cluster_min;
    int8_t halfw[ECB_MAX_EPS + 1];  // half width of the eps-disc at |dy|
    // exact-order mode: the emulated kd-tree is exported (one 16-byte node {pixel, left, right, parent} per point slot, same
    // indexing as pix[pol]) and every kept cluster whose median norm is tied is queued for k_bfs_order
    int exact_order;
    uint32_t *kd_nodes[2];
    BfsItem *bfs_items;
    unsigned *bfs_count;
    int bfs_cap;
};

struct BfsArgs {
    const BfsItem *items;
    const unsigned *count;      // device: number of items
    int max_items;
    const ProbDesc *prob;
    const uint32_t *pix[2];
    const int32_t *labels[2];
    const uint4 *kd_nodes[2];   // {pixel, left, right, parent}
    uint32_t *members[2];       // in: nothing required / out: member pids in BFS pop order at [off + mem_off, +size)
    uint32_t *scratch[2];       // same layout as members: unsorted frontier
    unsigned long long *key[2]; // per point slot
    int init_keys;              // 1: keys of the cluster's members are initialised here from the (ascending) member list
    KeptCluster *ktab;          // may be null
    int max_k;
    double eps;
};

size_t ecb_cluster_smem_bytes(int PW, int PH, int n_cap, int max_k, bool arrays_in_smem, bool rank32, bool st16);
// words per bitmap row: the padded sensor width W + 2E, rounded up to whole words (row_bits may read the word after a
// row's last one, but for x0 + len <= W + 2E only for bits it masks off; the word after the last row of U and C exists)
static inline int ecb_cluster_row_words(int W, int E) { return (W + 2 * E + 31) >> 5; }
int ecb_launch_cluster(ecb_ctx *ctx, ClusterArgs &a, int max_n);
int ecb_launch_bfs(ecb_ctx *ctx, BfsArgs &a);
// general points: the tree is {left, right, parent, depth << 1 | side} and coordinates come from P[n][dim] (ecb_gridhash.cu)
int ecb_launch_bfs_general(ecb_ctx *ctx, BfsArgs &a, const double *P, int dim);
// stable device sort of the loaded events (ev_t, ev_xyp) by time stamp: the reference's multimap load accepts any file order
int ecb_sort_events_by_time(ecb_ctx *ctx, int64_t n);
// DBSCAN::Run for any input (non-integer coordinates, duplicates, any eps, dim <= ECB_GH_MAXD): grid hash + radix sort
int ecb_dbscan_general(ecb_ctx *ctx, const double *pts, int dim, const int64_t *offsets, int n_problems, double eps,
                       uint32_t min_pts, int32_t *labels, int32_t *n_clusters, int32_t *cluster_sizes, uint32_t *members);
// every cluster of every problem -> BfsItem (ecb_dbscan_run_ordered): csize/cseed/coff are per point slot (index off + cid)
int ecb_launch_bfs_all_items(ecb_ctx *ctx, const ProbDesc *prob, const ProbHdr *hdr, int n_prob, const int32_t *labels,
                             uint32_t *csize, uint32_t *cseed, uint32_t *coff, BfsItem *items, unsigned *count, int cap);
