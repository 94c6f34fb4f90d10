// Shared device helpers and the context layout of libecb (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/eventcalib_b200.h"

#define ECB_MAX_EPS 15      // stencil rows fit a 64-bit funnel window (2*15+1 = 31 bits)
#define ECB_NONE 0xFFFFFFFFu
#define ECB_GH_MAXD 4       // largest point dimension of the general (grid-hash) DBSCAN path
#define ECB_GH_NBUF 32      // device buffers of that path

// packed event / pixel word:  x bits 0..14, y bits 15..29, bit 30 invalid, bit 31 polarity
#define ECB_PIX_X(p) ((p) & 0x7FFFu)
#define ECB_PIX_Y(p) (((p) >> 15) & 0x7FFFu)
#define ECB_PIX_POL(p) ((p) >> 31)
#define ECB_PIX_XY(p) ((p) & 0x3FFFFFFFu)
#define ECB_PIX_INVALID 0x40000000u

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct ecb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    uint64_t launches = 0;
    int sm_count = 148;
    int smem_optin = 0;
    int width = 0, height = 0;
    bool prof = false;
    // How the host waits for the stream (ECB_BLOCKING_SYNC, read at creation): 0 cudaStreamSynchronize (spins), 1 sleep on a
    // blocking event, 2 poll an event with sched_yield() in between — for many contexts / ranks on few host cores (8 ranks x 4
    // slice threads on a 32-core box starve each other when every wait spins)
    int sync_mode = 0;
    cudaEvent_t sync_ev = nullptr;
    cudaEvent_t pev[ECB_N_STAGES][2] = {};
    bool pev_used[ECB_N_STAGES] = {};

    // events (SoA)
    int64_t n_events = 0;
    DevBuf ev_raw, ev_t, ev_xyp, ev_flag;
    // front end
    int n_win = 0;
    ecb_frontend_params fp{};
    DevBuf win_t, win_lohi, win_ptoff, summary, arrive, pts[2], labels[2], scratch, ktab, kmem, cand, status, pair_tab;
    int max_k_auto = 128;     // kept-cluster table capacity of the automatic mode (max_clusters = 0): grows with the data, sticky
    std::vector<int64_t> h_lohi, h_ptoff;
    int64_t total_points = 0;
    int cand_stride = 0;
    // exact member order / medians (ecb_bfs.cu): exported kd-tree, claim keys, work items, frontier scratch
    DevBuf kd_tree, bfs_key, bfs_items, bfs_front, bfs_tab;
    // k_uset_order: std::hash<double> of every integer coordinate of the sensor (+ the hash_combine constant)
    DevBuf ord_htab;
    int ord_htab_n = 0;
    // dbscan boundary
    DevBuf db_pix, db_off, db_labels, db_hdr, db_scratch, db_dims, db_hdr_b, db_ktab, db_counter;
    DevBuf gh[ECB_GH_NBUF];   // general path (ecb_gridhash.cu)
    // fit
    DevBuf fit_in, fit_off, fit_out;
    // pinned staging (device -> host), and mapped pinned staging the device pulls small uploads from
    void *pinned = nullptr;
    size_t pinned_cap = 0;
    void *up = nullptr;
    size_t up_cap = 0, up_off = 0;
    // cost evaluation (ecb_cost.cu)
    void *cost = nullptr;
    // covariance workspace (ecb_lmdev.cu), kept for repeated calls with the same spline layout
    void *cov = nullptr;
    // incremented by ecb_cost_setup, ecb_cost_set_rotation_model and a change of const_intrinsics: a covariance computed before
    // refers to other knots, another rotation tangent or other free parameters
    uint64_t spline_gen = 0;
    // intrinsics held constant in the spline stage (ecb_cost_set_constant_intrinsics): bit i = intrinsic i (fx fy cx cy k1 .. k5)
    uint32_t const_intrinsics = 0;
    // staging of the host variant of ecb_pose_covariance (ecb_pose_cov.cu)
    DevBuf pose_io;
    // control points, count and host staging of ecb_trajectory_motion / ecb_motion_covariance (ecb_pose_cov.cu)
    DevBuf motion_io;
    // control points, samples, partial sums and residuals of ecb_gyro_calibrate (ecb_gyro.cu)
    DevBuf gyro_io;
    // incremented by every event load: the residual report by key frame needs the events its association read
    uint64_t events_gen = 0;
};

// the splines of ecb_cost_setup on the device (ecb_cost.cu); ECB_ERR_STATE before the setup
struct EcbSplineView {
    const double *knots;
    const int *knot_off, *ncp, *cp_off;
    int n_splines, total_cp, so3;
    // the first segment whose knot range holds u (EventCalibSpline::time2splineIdx; NaN holds in no range), with *kn its knots
    // and *nk their count; -1 when there is none
    __device__ __forceinline__ int segment(double u, const double **kn, int *nk) const {
        for (int s = 0; s < n_splines; ++s) {
            *kn = knots + knot_off[s];
            *nk = ncp[s] + 4;
            if (u >= (*kn)[0] && u <= (*kn)[*nk - 1]) return s;
        }
        return -1;
    }
};
extern "C" int ecb_cost_spline_view(ecb_ctx *ctx, EcbSplineView *v);
// the result of the last successful ecb_covariance (ecb_lmdev.cu): the band of Z (layout of cov_band), the point x
// (intrinsics 9 | rotation 4C | translation 3C), the rotation model and ctx->spline_gen at that call; ECB_ERR_STATE without one
struct EcbCovView {
    const double *Zb, *x;
    int total_cp, so3;
    uint64_t spline_gen;
};
extern "C" int ecb_covariance_view(ecb_ctx *ctx, EcbCovView *v);

// Constant intrinsics: the reduced problem of a Ceres SubsetManifold on the intrinsics block.  Once the packed normal equations
// are assembled, the row and column of J^T J and the entry of J^T r of every constant intrinsic are zeroed; the Jacobi scale, the
// clamped LM diagonal, the zero step component and the zero projected gradient follow from the unchanged LM code.  Entry (ri, ci)
// of the assembled system or of the covariance: ri / ci = intrinsic index of its row / column, -1 for a control-point row or
// column (and for the column of J^T r).  Mask 0 passes every entry unchanged.
#define ECB_ALL_INTRINSICS 0x1FFu
#ifdef __CUDACC__
__host__ __device__ __forceinline__
#else
inline
#endif
double ecb_zero_constant(uint32_t mask, int ri, int ci, double v) {
    return ((ri >= 0 && ((mask >> ri) & 1u)) || (ci >= 0 && ((mask >> ci) & 1u))) ? 0.0 : v;
}

// Stable LSD radix sort (ecb_gridhash.cu) of (key, idx) pairs by the low `bits` bits of key, 8 bits per pass, n >= 1 and
// n < 2^32; the result ends in key[*res] / idx[*res] (ping-pong buffers 0 / 1).  hist: gh_radix_hist_bytes(n) bytes.
int gh_radix_sort(ecb_ctx *ctx, uint64_t *key[2], uint32_t *idx[2], int64_t n, int bits, uint32_t *hist, int *res);
size_t gh_radix_hist_bytes(int64_t n);

int ecb_fail(ecb_ctx *ctx, int code, const char *fmt, ...);
int ecb_reserve(ecb_ctx *ctx, DevBuf &b, size_t bytes);
int ecb_check(ecb_ctx *ctx, cudaError_t e, const char *what);
cudaError_t ecb_stream_sync(ecb_ctx *ctx);  // wait for the context's stream (spinning or sleeping, see blocking_sync)
int ecb_d2h(ecb_ctx *ctx, void *dst, const void *src, size_t bytes);  // pinned-staged copy + stream sync
// Small host -> device upload that does not touch the copy engines: the data is staged in mapped pinned memory and a
// kernel on the context stream pulls it over PCIe, so it cannot queue behind another context's bulk record upload.
int ecb_h2d(ecb_ctx *ctx, void *dst, const void *src, size_t bytes);
#define ECB_CUDA(ctx, call)                                   \
    do {                                                      \
        int _rc = ecb_check((ctx), (call), #call);            \
        if (_rc) return _rc;                                  \
    } while (0)
#define ECB_LAUNCHED(ctx) ((ctx)->launches++)
// stage timing: ECB_PROF_BEGIN/END bracket a kernel launch with events when profiling is on
#define ECB_PROF_BEGIN(ctx, st) do { if ((ctx)->prof) cudaEventRecord((ctx)->pev[st][0], (ctx)->stream); } while (0)
#define ECB_PROF_END(ctx, st) do { if ((ctx)->prof) { cudaEventRecord((ctx)->pev[st][1], (ctx)->stream); (ctx)->pev_used[st] = true; } } while (0)

// ---------------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v) {
    const unsigned lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= (unsigned) o) v += t;
    }
    return v;
}

// Block-wide exclusive scan of one value per thread; returns the exclusive prefix, *total = block sum.
// `ws` is a shared array of at least 33 words. All threads of the block must call it.
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *ws, uint32_t *total) {
    const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    uint32_t inc = warp_incl_scan(v);
    __syncthreads();  // protect ws from a previous use
    if (lane == 31) ws[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = lane < nw ? ws[lane] : 0;
        uint32_t wi = warp_incl_scan(w);
        ws[lane] = wi - w;
        if (lane == 31) ws[32] = wi;
    }
    __syncthreads();
    *total = ws[32];
    return ws[wid] + inc - v;
}

// bits [x0, x0+len) of a bitmap row (len <= 32); reads the word after x0's, which must be readable (it only supplies bits
// when x0 + len crosses into it)
__device__ __forceinline__ uint32_t row_bits(const uint32_t *row, int x0, int len) {
    const int wi = x0 >> 5, sh = x0 & 31;
    uint64_t v = (uint64_t) row[wi] | ((uint64_t) row[wi + 1] << 32);
    return (uint32_t) (v >> sh) & (len >= 32 ? 0xFFFFFFFFu : ((1u << len) - 1u));
}
__device__ __forceinline__ uint32_t test_bit(const uint32_t *row, int x) { return (row[x >> 5] >> (x & 31)) & 1u; }
#endif
