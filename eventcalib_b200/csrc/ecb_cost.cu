// Cost evaluation of the dynamic-calibration objective on the GPU.
//
//   k_associate_*   EventCalibSpline::optimize association loop (src/EventCalibSpline.cpp:157-192) + findCenter
//                   (include/.../CirclesEventFrame.hpp:50-65): raw event -> nearest keyframe in time -> nearest circle
//                   -> | ||p-c|| - r | < 5 px -> residual record (ordered compaction, two passes)
//   k_prepare       findSpan + dersBasisFuns per residual (core/spline/.../BsplineReal.hpp:208-231,107-145); the basis
//                   is constant over the LM iterations, so it is computed once here
//   k_normal_eq     residual + closed-form Jacobian (ecb_residual.h) per lane, then the per-span Gram matrix
//                   [J | r]^T [J | r] (34 x 34, padded to 40) on the FP64 tensor pipe: mma.sync m8n8k4 f64 (DMMA),
//                   15 upper 8x8 tiles per warp kept in registers, J staged through shared memory transposed
//                   (conflict-free for both the lane-per-residual stores and the fragment loads).
//                   B200 measured: DMMA 37.0 TFLOP/s == DFMA 36.4 TFLOP/s (profiles/r1_fp64_peak.txt), so the
//                   tensor path costs nothing in peak and removes the shared-memory/issue bottleneck of a
//                   CUDA-core register-tiled SYRK.  tcgen05 has no f64 kind.
//   k_reduce_*      fixed-order reduction of the per-work-item partials -> run-to-run identical J^T J / J^T r / cost
//   k_cost          cost-only evaluation (LM step acceptance)
//   k_record_report, k_group_*        the residual report (board units) and the same fit in pixels (forward model of
//                                     ecb_camera.h): one value per record, then statistics per group
//   k_keyframe_reproj                 the key frames' circle centres reprojected at their stamps
//   k_reject_count, k_reject_write    outlier rejection: ordered compaction of the records that are kept (ecb_cost_reject)
//   k_reassoc_count the association's pass 1 through the calibrated model (ecb_cost_reassociate); pass 2 is k_assoc_write
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "ecb_bspline.cuh"
#include "ecb_camera.h"
#include "ecb_common.cuh"
#include "ecb_residual_so3.h"

namespace {

constexpr int NE_THREADS = 256;            // 8 warps
constexpr int NE_WARPS = NE_THREADS / 32;
constexpr int TILE_ROWS = 34, TILE_LD = 36;  // [param | r][residual], LD % 16 == 4 -> conflict-free fragment loads
constexpr int N_TILES = 10;                 // upper 8x8 DMMA tiles of the leading 32x32 block of the 34x34 Gram matrix
// per work item: 10 tiles | row 32 (32) | row 33 = J^T r (32) | H[32][32], g[32], sum r^2, cost
constexpr int PART_E32 = N_TILES * 64, PART_E33 = PART_E32 + 32, PART_SC = PART_E33 + 32, PART_STRIDE = PART_SC + 8;
constexpr int CHUNK = 2048;                 // residuals per work item
constexpr int OUT_STRIDE = 33 * 33 + 33;    // per span: H (full symmetric) | g

struct CostState {
    int n_splines = 0, total_cp = 0, total_spans = 0;
    std::vector<int> n_cp, cp_off, span_off, knot_off;
    std::vector<double> knots;
    double radius = 1.75, huber = 0.35;
    bool use_circ = false;  // residuals carry a landmark index (association path) instead of explicit landmark coordinates
    int so3 = 0;  // rotation model: 0 normalised quaternion spline (useSO3: 0), 1 cumulative SO(3) spline (useSO3: 1)
    int64_t n_res = 0;
    int n_items = 0;
    DevBuf d_knots, d_knot_off, d_ncp, d_cp_off, d_span_off;
    DevBuf obs, lm, tt, spl, basis, cp0, span;        // residual records (SoA)
    DevBuf span_start, items, part, out, params, cost_part, flags;
    DevBuf ev_flag, ev_cnt, ev_tag, kf_t, kf_circ, kf_c32, lm_tab, sel_event, sel_circle;
    std::vector<int64_t> h_span_start;
    // the records come from an association (event_index / circle_id exist) over K key frames, n_circ circles, and the events of
    // ctx->events_gen == assoc_events_gen
    bool assoc = false;
    int assoc_K = 0, assoc_n_circ = 0;
    uint64_t assoc_events_gen = 0;
    // what ecb_cost_reassociate reuses of the association: its stamps (st->kf_t, or the caller's device table) and window
    const double *assoc_kf_t = nullptr;
    double assoc_gate2 = 0.0;
    DevBuf rep_r, rep_key[2], rep_idx[2], rep_hist, rep_start, rep_out, rep_kf;  // residual report (ecb_cost_residual_groups)
    DevBuf rep_io;  // reprojection report: invalid count; staging of ecb_keyframe_reprojection
    // ecb_cost_reject: the spare set of record buffers the kept records are compacted into, then swapped with the live ones
    // (order of reject_bufs)
    DevBuf rej[9];
    uint64_t xch_last_epoch = 0;   // ecb_cost_normal_eq_exchange: last epoch sent / generation of the caller's sequence
    uint32_t xch_generation = 0;
};

CostState *state(ecb_ctx *ctx) {
    if (!ctx->cost) ctx->cost = new CostState();
    return (CostState *) ctx->cost;
}

// ------------------------------------------------------------------------------------ prepare ----
__global__ void k_prepare(const double *__restrict__ t, const int *__restrict__ spl, int64_t n, const double *__restrict__ knots,
                          const int *__restrict__ knot_off, const int *__restrict__ ncp, const int *__restrict__ cp_off,
                          const int *__restrict__ span_off, double *__restrict__ basis, int *__restrict__ cp0,
                          int *__restrict__ span, uint32_t *__restrict__ flags) {
    const int64_t k = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int s = spl[k];
    const double *kn = knots + knot_off[s];
    const int nk = ncp[s] + 4;
    const double u = t[k];
    if (!(u >= kn[0] && u <= kn[nk - 1])) {  // outside the spline: the reference never creates such a block
        atomicOr(flags, 1u);
        span[k] = 0;
        cp0[k] = 0;
        return;
    }
    const int sp = find_span_dev(kn, nk, u);
    double N[4];
    basis_dev(kn, sp, u, N);
    reinterpret_cast<double4 *>(basis)[k] = make_double4(N[0], N[1], N[2], N[3]);
    cp0[k] = cp_off[s] + sp - 3;
    const int gs = span_off[s] + sp - 3;
    span[k] = gs;
    if (k > 0) {  // records must be ordered by (spline, time) so that spans are contiguous
        const int sprev = spl[k - 1];
        if (sprev > s || (sprev == s && t[k - 1] > u)) atomicOr(flags, 2u);
    }
}

__global__ void k_span_start(const int *__restrict__ span, int64_t n, int n_spans, int64_t *__restrict__ start) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s > n_spans) return;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        int64_t m = (lo + hi) >> 1;
        if (span[m] < s) lo = m + 1; else hi = m;
    }
    start[s] = lo;
}

// ---------------------------------------------------------------------------------- normal eq ----
struct Item {
    int64_t begin, end;
    int span, pad;
};

struct NeArgs {
    const double *obs, *lm, *basis;
    const int *circ;        // landmark index per residual into lm_tab (association path), or null: explicit `lm` per residual
    const double *lm_tab;
    const int *cp0;
    const Item *items;
    int n_items;
    const double *params;  // intr[9] | rot[4*C] | trans[3*C]
    int total_cp;
    double radius, huber;
    double *part;
    const int *go;         // device flag (may be null): 0 = the launch is a no-op (device-side LM loop: step rejected / finished)
};

// the residual records (SoA) as the evaluation kernels read them: record k's first control point c0, basis b, observation o
// and landmark L (lm_tab[circ[k]] on the association path, else the explicit lm[3k])
struct RecordView {
    const double *obs, *lm;
    const int *circ;
    const double *lm_tab, *basis;
    const int *cp0;
    __device__ __forceinline__ void load(int64_t k, int &c0, double b[4], double2 &o, double L[3]) const {
        c0 = cp0[k];
        const double4 b4 = reinterpret_cast<const double4 *>(basis)[k];
        b[0] = b4.x, b[1] = b4.y, b[2] = b4.z, b[3] = b4.w;
        o = reinterpret_cast<const double2 *>(obs)[k];
        const double *p = circ ? lm_tab + 3 * circ[k] : lm + 3 * k;
        L[0] = p[0], L[1] = p[1], L[2] = p[2];
    }
};

__device__ __forceinline__ void dmma(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

template <int MINB, bool SO3>
__global__ void __launch_bounds__(NE_THREADS, MINB) k_normal_eq(const NeArgs a) {
    extern __shared__ __align__(16) double sm_tiles[];
    if (a.go && *a.go == 0) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    double *tile = sm_tiles + (size_t) wid * TILE_ROWS * TILE_LD;
    const int g = lane >> 2, t = lane & 3;
    const double *intr = a.params, *rot = a.params + 9, *trans = a.params + 9 + 4 * (size_t) a.total_cp;
    const int gw = blockIdx.x * NE_WARPS + wid, nw = gridDim.x * NE_WARPS;
    for (int it = gw; it < a.n_items; it += nw) {
        const Item item = a.items[it];
        // Gram matrix of [J | r] (34 columns): the leading 32x32 block on the FP64 tensor pipe (10 upper 8x8 tiles),
        // rows 32 (last parameter) and 33 (r) with plain DFMAs — padding 34 -> 40 would waste 5 of 15 DMMA tiles
        double acc[N_TILES][2];
#pragma unroll
        for (int i = 0; i < N_TILES; ++i) acc[i][0] = acc[i][1] = 0.0;
        double e32 = 0.0, e33 = 0.0;            // lane j: sum_k J_k[32] J_k[j], sum_k r_k J_k[j]
        double s3232 = 0.0, s3233 = 0.0, s3333 = 0.0, cost = 0.0;  // per-lane partials over its own residuals
        for (int64_t base = item.begin; base < item.end; base += 32) {
            const int64_t k = base + lane;
            double res = 0.0;
            __syncwarp();  // the previous group's fragment loads are done
            if (k < item.end) {
                int c0;
                double b[4], L[3];
                double2 o;
                RecordView{a.obs, a.lm, a.circ, a.lm_tab, a.basis, a.cp0}.load(k, c0, b, o, L);
                // the Jacobian is scattered straight into column `lane` of the shared tile (no register array)
                const EcbResidualOut r =
                    SO3 ? ecb_residual_so3<true, TILE_LD>(intr, rot + 4 * (size_t) c0, trans + 3 * (size_t) c0, b, o.x, o.y,
                                                          L[0], L[1], L[2], a.radius, a.huber,
                                                          tile + lane)
                        : ecb_residual<true, TILE_LD>(intr, rot + 4 * (size_t) c0, trans + 3 * (size_t) c0, b, o.x, o.y,
                                                      L[0], L[1], L[2], a.radius, a.huber,
                                                      tile + lane);
                res = r.res;
                cost += r.cost;
            } else {
#pragma unroll
                for (int c = 0; c < 33; ++c) tile[c * TILE_LD + lane] = 0.0;
            }
            tile[33 * TILE_LD + lane] = res;
            __syncwarp();
            {
                const double x32 = tile[32 * TILE_LD + lane];
                s3232 += x32 * x32;
                s3233 += x32 * res;
                s3333 += res * res;
            }
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
                double f[4];
#pragma unroll
                for (int G = 0; G < 4; ++G) f[G] = tile[(8 * G + g) * TILE_LD + 4 * ks + t];
                int ti = 0;
#pragma unroll
                for (int I = 0; I < 4; ++I)
#pragma unroll
                    for (int Jt = I; Jt < 4; ++Jt) {
                        dmma(acc[ti][0], acc[ti][1], f[I], f[Jt]);
                        ++ti;
                    }
                // rows 32 / 33: lane j accumulates column j; residual index rotated per lane group -> conflict-free loads
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int kk = (4 * ks + q + (lane >> 2)) & 31;
                    const double aj = tile[lane * TILE_LD + kk];
                    e32 += aj * tile[32 * TILE_LD + kk];
                    e33 += aj * tile[33 * TILE_LD + kk];
                }
            }
        }
        // partial of this work item
        double *p = a.part + (size_t) it * PART_STRIDE;
#pragma unroll
        for (int ti = 0; ti < N_TILES; ++ti) reinterpret_cast<double2 *>(p + ti * 64)[lane] = make_double2(acc[ti][0], acc[ti][1]);
        p[PART_E32 + lane] = e32;
        p[PART_E33 + lane] = e33;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            cost += __shfl_xor_sync(0xffffffffu, cost, o);
            s3232 += __shfl_xor_sync(0xffffffffu, s3232, o);
            s3233 += __shfl_xor_sync(0xffffffffu, s3233, o);
            s3333 += __shfl_xor_sync(0xffffffffu, s3333, o);
        }
        if (lane == 0) {
            p[PART_SC + 0] = s3232;
            p[PART_SC + 1] = s3233;
            p[PART_SC + 2] = s3333;
            p[PART_SC + 3] = cost;
        }
    }
}

// out[s] = sum over the span's work items, fixed order; tiles -> full symmetric 33x33 + gradient
__global__ void k_reduce_spans(const double *__restrict__ part, const int *__restrict__ item_start, int n_spans,
                               double *__restrict__ out, const int *__restrict__ go = nullptr) {
    const int s = blockIdx.x;
    if (s >= n_spans || (go && *go == 0)) return;
    const int i0 = item_start[s], i1 = item_start[s + 1];
    double *o = out + (size_t) s * OUT_STRIDE;
    for (int e = threadIdx.x; e < PART_SC + 2; e += blockDim.x) {
        double v = 0.0;
        for (int it = i0; it < i1; ++it) v += part[(size_t) it * PART_STRIDE + e];
        if (e < PART_E32) {
            const int ti = e >> 6, r = (e >> 3) & 7, c = e & 7;
            int I = 0, rem = ti;  // tile index -> (I, Jt), I <= Jt over 4 groups
            while (rem >= 4 - I) {
                rem -= 4 - I;
                ++I;
            }
            const int Jt = I + rem;
            const int i = 8 * I + r, j = 8 * Jt + c;
            if (I != Jt || i <= j) {
                o[i * 33 + j] = v;
                o[j * 33 + i] = v;
            }
        } else if (e < PART_E33) {
            const int j = e - PART_E32;
            o[32 * 33 + j] = v;
            o[j * 33 + 32] = v;
        } else if (e < PART_SC) {
            o[1089 + (e - PART_E33)] = v;
        } else if (e == PART_SC) {
            o[32 * 33 + 32] = v;
        } else {
            o[1089 + 32] = v;
        }
    }
}

// ---------------------------------------------------------------- fused reduce + inter-GPU exchange ----
// Multi-GPU normal equations without a separate collective: the span reduction of every rank stores its result straight
// into a slot of EVERY peer's receive buffer over NVLink (peer-mapped memory), a one-warp kernel publishes
// (epoch, span range, cost) to the peers, and each rank sums the slots in rank order once all have arrived — a one-shot
// all-reduce whose send side is the epilogue of k_reduce_spans.  Deterministic (fixed rank order), identical on every
// rank, double-buffered by epoch parity (a rank can be at most one exchange ahead of a peer).
//
// receive buffer of one rank:  [parity 0 | parity 1],  parity block = n_ranks slots,  slot = header (8 doubles:
// epoch as u64, first span, last span, cost) + total_spans * OUT_STRIDE doubles (only [first, last] are written).
constexpr int XH = 8;  // header doubles

__host__ __device__ inline size_t xslot_doubles(int total_spans) { return (size_t) XH + (size_t) total_spans * OUT_STRIDE; }

struct XPeers {
    double *base[ECB_MAX_PEERS];
    int n_ranks, rank;
};

// Where an exchange lives in the receive buffers: the epoch comes from the host (ecb_cost_normal_eq_exchange) or from a device
// counter (device-side LM loop, ecb_lmdev.cu: the host enqueues many iterations ahead and does not know which of them exchange).
struct XCtl {
    const int *go;                        // device flag (may be null): 0 = no-op
    const unsigned long long *d_epoch;    // device epoch counter, or null: use `epoch`
    unsigned long long epoch;
    size_t slot;                          // doubles per slot
    int n_ranks, rank;
    __device__ __forceinline__ unsigned long long e() const { return d_epoch ? *d_epoch : epoch; }
    __device__ __forceinline__ size_t parity_off() const { return (size_t) (e() & 1ull) * (size_t) n_ranks * slot; }
    __device__ __forceinline__ size_t my_slot_off() const { return parity_off() + (size_t) rank * slot; }
};

// k_reduce_spans whose stores go to the slot of this rank in every peer's buffer
__global__ void k_reduce_spans_push(const double *__restrict__ part, const int *__restrict__ item_start, int span_lo, int span_hi,
                                    XPeers peers, XCtl x) {
    const int s = span_lo + blockIdx.x;
    if (s > span_hi || (x.go && *x.go == 0)) return;
    const size_t slot_off = x.my_slot_off();
    const int i0 = item_start[s], i1 = item_start[s + 1];
    for (int e = threadIdx.x; e < PART_SC + 2; e += blockDim.x) {
        double v = 0.0;
        for (int it = i0; it < i1; ++it) v += part[(size_t) it * PART_STRIDE + e];
        int a0 = -1, a1 = -1;  // the (at most two, symmetric) destinations inside the span block
        if (e < PART_E32) {
            const int ti = e >> 6, r = (e >> 3) & 7, c = e & 7;
            int I = 0, rem = ti;
            while (rem >= 4 - I) {
                rem -= 4 - I;
                ++I;
            }
            const int Jt = I + rem;
            const int i = 8 * I + r, j = 8 * Jt + c;
            if (I != Jt || i <= j) {
                a0 = i * 33 + j;
                a1 = j * 33 + i;
            }
        } else if (e < PART_E33) {
            const int j = e - PART_E32;
            a0 = 32 * 33 + j;
            a1 = j * 33 + 32;
        } else if (e < PART_SC) {
            a0 = 1089 + (e - PART_E33);
        } else if (e == PART_SC) {
            a0 = 32 * 33 + 32;
        } else {
            a0 = 1089 + 32;
        }
        if (a0 < 0) continue;
        for (int p = 0; p < peers.n_ranks; ++p) {
            double *o = peers.base[p] + slot_off + XH + (size_t) s * OUT_STRIDE;
            o[a0] = v;
            if (a1 >= 0) o[a1] = v;
        }
    }
}

// after the pushes (stream order): publish this rank's header to every peer
__global__ void k_exchange_signal(XPeers peers, XCtl x, int span_lo, int span_hi, const double *__restrict__ cost) {
    const int p = threadIdx.x;
    if (p >= peers.n_ranks || (x.go && *x.go == 0)) return;
    double *h = peers.base[p] + x.my_slot_off();
    h[1] = (double) span_lo;
    h[2] = (double) span_hi;
    h[3] = *cost;
    __threadfence_system();
    *reinterpret_cast<volatile unsigned long long *>(h) = x.e();
}

// one warp: wait until every rank's header of this parity carries the epoch.  The spin is bounded (ECB_EXCHANGE_TIMEOUT_S
// seconds, default 30: lazy module loads or host pauses of a peer process must not trip it) and a timeout raises a sticky
// error bit per rank that k_exchange_sum turns into a NaN cost, so no caller can mistake a partial sum for a result.
__global__ void k_exchange_wait(const double *__restrict__ recv, XCtl x, long long timeout_clocks, unsigned *err) {
    const int r = threadIdx.x;
    if (r >= x.n_ranks || (x.go && *x.go == 0)) return;
    const unsigned long long epoch = x.e();
    const volatile unsigned long long *f =
        reinterpret_cast<const volatile unsigned long long *>(recv + x.parity_off() + (size_t) r * x.slot);
    const long long t0 = clock64();
    while (*f != epoch) {
        if (clock64() - t0 > timeout_clocks) {
            atomicOr(err, 1u << r);
            break;
        }
        __nanosleep(200);
    }
    __threadfence_system();
}

// out[s] = sum over the ranks whose range holds s, in rank order; out[n_spans*OUT_STRIDE] = sum of the costs
__global__ void k_exchange_sum(const double *__restrict__ recv, XCtl x, int n_spans, double *__restrict__ out,
                               const unsigned *__restrict__ err) {
    const int s = blockIdx.x;
    if (x.go && *x.go == 0) return;
    const size_t parity_off = x.parity_off(), slot_stride = x.slot;
    const int n_ranks = x.n_ranks;
    if (s == n_spans) {
        if (threadIdx.x == 0) {
            double c = 0.0;
            for (int r = 0; r < n_ranks; ++r) c += recv[parity_off + (size_t) r * slot_stride + 3];
            if (err && *err) c = __longlong_as_double(0x7FF8000000000000ll);  // a rank never arrived: no result
            out[(size_t) n_spans * OUT_STRIDE] = c;
            out[(size_t) n_spans * OUT_STRIDE + 1] = 0.0;
        }
        return;
    }
    for (int e = threadIdx.x; e < OUT_STRIDE; e += blockDim.x) {
        double v = 0.0;
        for (int r = 0; r < n_ranks; ++r) {
            const double *slot = recv + parity_off + (size_t) r * slot_stride;
            if (s >= (int) slot[1] && s <= (int) slot[2]) v += slot[XH + (size_t) s * OUT_STRIDE + e];
        }
        out[(size_t) s * OUT_STRIDE + e] = v;
    }
}

// Scalar all-reduce over the same peer buffers (device-side LM loop: the candidate cost of every iteration): rank r stores
// (value, epoch) into slot r of every peer's scalar area, waits for all slots of this epoch and adds them in rank order.
// One warp; *value is replaced by the sum.  The scalar area follows the two parity blocks of the span slots.
__global__ void k_exchange_scalar(XPeers peers, XCtl x, size_t scalar_off, double *value, long long timeout_clocks, unsigned *err) {
    const int p = threadIdx.x;
    if (x.go && *x.go == 0) return;
    const unsigned long long epoch = x.e();
    const size_t par = scalar_off + (size_t) (epoch & 1ull) * 2 * (size_t) x.n_ranks;
    if (p < x.n_ranks) {
        double *h = peers.base[p] + par + 2 * (size_t) x.rank;
        h[1] = *value;
        __threadfence_system();
        *reinterpret_cast<volatile unsigned long long *>(h) = epoch;
        const volatile unsigned long long *f = reinterpret_cast<const volatile unsigned long long *>(peers.base[x.rank] + par + 2 * (size_t) p);
        const long long t0 = clock64();
        while (*f != epoch) {
            if (clock64() - t0 > timeout_clocks) {
                atomicOr(err, 1u << p);
                break;
            }
            __nanosleep(100);
        }
        __threadfence_system();
    }
    __syncwarp();
    if (p == 0) {
        double c = 0.0;
        for (int r = 0; r < x.n_ranks; ++r) c += *reinterpret_cast<const volatile double *>(peers.base[x.rank] + par + 2 * (size_t) r + 1);
        if (*err) c = __longlong_as_double(0x7FF8000000000000ll);
        *value = c;
    }
}

__global__ void k_reduce_cost(const double *__restrict__ part, int n, int stride, int offset, double *__restrict__ out,
                              const int *__restrict__ go = nullptr) {
    // single block, fixed order: thread-strided partial sums, then a shared-memory tree
    __shared__ double sh[256];
    if (go && *go == 0) return;
    double v = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) v += part[(size_t) i * stride + offset];
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = sh[0];
}

template <bool SO3, int MINB>
__global__ void __launch_bounds__(256, MINB) k_cost(const double *__restrict__ obs, const double *__restrict__ lm,
                                             const int *__restrict__ circ, const double *__restrict__ lm_tab,
                                             const double *__restrict__ basis, const int *__restrict__ cp0, int64_t n,
                                             const double *__restrict__ params, int total_cp, double radius, double huber,
                                             double *__restrict__ block_part, const int *__restrict__ go = nullptr) {
    __shared__ double sh[256];
    if (go && *go == 0) return;
    const double *intr = params, *rot = params + 9, *trans = params + 9 + 4 * (size_t) total_cp;
    double c = 0.0;
    const RecordView rv{obs, lm, circ, lm_tab, basis, cp0};
    for (int64_t k = (int64_t) blockIdx.x * 256 + threadIdx.x; k < n; k += (int64_t) gridDim.x * 256) {
        int c0;
        double b[4], L[3];
        double2 o;
        rv.load(k, c0, b, o, L);
        c += SO3 ? ecb_residual_so3<false>(intr, rot + 4 * (size_t) c0, trans + 3 * (size_t) c0, b, o.x, o.y, L[0], L[1], L[2],
                                           radius, huber, nullptr).cost
                 : ecb_residual<false>(intr, rot + 4 * (size_t) c0, trans + 3 * (size_t) c0, b, o.x, o.y, L[0], L[1], L[2], radius,
                                       huber, nullptr).cost;
    }
    sh[threadIdx.x] = c;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) block_part[blockIdx.x] = sh[0];
}

// -------------------------------------------------------------------------------- association ----
struct AssocArgs {
    const double *ev_t;
    const uint32_t *ev_xyp;
    int64_t n_ev;
    const double *knots;
    const int *knot_off, *ncp;
    int n_splines;
    const double *kf_t, *kf_circ, *lm_tab;
    const float2 *kf_c32;  // FP32 copy of the circle centres, row stride n_circ32 (even), absent / padding = far away
    int K, n_circ, n_circ32;
    double gate2;  // (5 step)^2
    // fused k_prepare (spline ranges sorted and disjoint): span / basis / first control point written with the record
    const int *cp_off, *span_off;
    double *basis;
    int *cp0, *span;
};

// the first spline segment whose knot range holds u, or -1
__device__ __forceinline__ int segment_of(const AssocArgs &a, double u) {
    for (int q = 0; q < a.n_splines; ++q) {
        const double *kn = a.knots + a.knot_off[q];
        if (u >= kn[0] && u <= kn[a.ncp[q] + 3]) return q;
    }
    return -1;
}

// returns the spline index and the circle id (or -1) of one raw event
__device__ __forceinline__ int assoc_one(const AssocArgs &a, int64_t i, int *spline_out) {
    const double u = a.ev_t[i];
    const int s = segment_of(a, u);
    if (s < 0) return -1;
    *spline_out = s;
    int lo = 0, hi = a.K;  // lower_bound over keyframe times
    while (lo < hi) {
        const int m = (lo + hi) >> 1;
        if (a.kf_t[m] < u) lo = m + 1; else hi = m;
    }
    int best = lo < a.K ? lo : a.K - 1;
    if (lo > 0 && (lo >= a.K || (u - a.kf_t[lo - 1]) <= (a.kf_t[lo] - u))) best = lo - 1;
    const double dt = u - a.kf_t[best];
    if (!(__dmul_rn(dt, dt) < a.gate2)) return -1;
    const uint32_t e = a.ev_xyp[i];
    if (e & ECB_PIX_INVALID) return -1;
    const double x = (double) ECB_PIX_X(e), y = (double) ECB_PIX_Y(e);
    const double *c = a.kf_circ + (size_t) best * a.n_circ * 3;
    int bi = -1;
    double bd = 0.0;
    // Nearest centre: FP32 preselection over all circles with sortable keys (distance bits | circle index), keeping the two
    // smallest.  When the runner-up is clearly farther than the winner the exact FP64 distance is evaluated for the winner
    // alone; near-ties (and nothing else) take the exact FP64 loop, so the result is the exact arg-min either way.
    {
        const float xf = (float) ECB_PIX_X(e), yf = (float) ECB_PIX_Y(e);  // pixel coordinates are exact in FP32
        const float4 *c4 = reinterpret_cast<const float4 *>(a.kf_c32 + (size_t) best * a.n_circ32);
        uint32_t k1 = 0xFFFFFFFFu, k2 = 0xFFFFFFFFu;
#pragma unroll 6
        for (int q = 0; q < a.n_circ32; q += 2) {
            const float4 cc = c4[q >> 1];
            const float dx0 = xf - cc.x, dy0 = yf - cc.y, dx1 = xf - cc.z, dy1 = yf - cc.w;
            const uint32_t ka = (__float_as_uint(fmaf(dx0, dx0, dy0 * dy0)) & 0xFFFFFF00u) | (uint32_t) q;
            const uint32_t kb = (__float_as_uint(fmaf(dx1, dx1, dy1 * dy1)) & 0xFFFFFF00u) | (uint32_t) (q + 1);
            k2 = min(k2, max(ka, k1));
            k1 = min(k1, ka);
            k2 = min(k2, max(kb, k1));
            k1 = min(k1, kb);
        }
        const float d1 = __uint_as_float(k1 & 0xFFFFFF00u), d2 = __uint_as_float(k2 | 0xFFu);
        if (d2 > d1 * 1.0001f + 0.02f) {  // unambiguous (FP32 error <= 2e-7 d + 3e-4 |d|^(1/2), key quantisation 1.5e-5 d)
            bi = (int) (k1 & 0xFFu);
            if (bi >= a.n_circ || c[3 * bi + 2] < 0) return -1;  // only absent circles
            const double dx = x - c[3 * bi], dy = y - c[3 * bi + 1];
            bd = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
        } else {
            for (int q = 0; q < a.n_circ; ++q) {
                if (c[3 * q + 2] < 0) continue;
                const double dx = x - c[3 * q], dy = y - c[3 * q + 1];
                const double dd = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
                if (bi < 0 || dd < bd) {
                    bi = q;
                    bd = dd;
                }
            }
        }
    }
    if (bi < 0) return -1;
    if (!(fabs(sqrt(bd) - c[3 * bi + 2]) < 5.0)) return -1;
    return bi;
}

constexpr int AS_THREADS = 256;

// FP32 copy of the circle centres for the preselection in assoc_one: rows padded to an even count; absent circles (r < 0)
// and padding sit at (3e18, 3e18) so they never win against a real circle
__global__ void k_circ32(const double *__restrict__ c, int K, int n_circ, int n_circ32, float2 *__restrict__ o) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K * n_circ32) return;
    const int k = i / n_circ32, q = i - k * n_circ32;
    float2 v = make_float2(3e18f, 3e18f);
    if (q < n_circ) {
        const double *p = c + ((size_t) k * n_circ + q) * 3;
        if (!(p[2] < 0)) v = make_float2((float) p[0], (float) p[1]);
    }
    o[i] = v;
}

// nearest key frame in time, ties -> the earlier frame (1-NN over the stamps, EventCalibSpline.cpp:166)
__device__ __forceinline__ int nearest_kf(const double *kf_t, int K, double u) {
    int lo = 0, hi = K;
    while (lo < hi) {
        const int m = (lo + hi) >> 1;
        if (kf_t[m] < u) lo = m + 1; else hi = m;
    }
    int best = lo < K ? lo : K - 1;
    if (lo > 0 && (lo >= K || (u - kf_t[lo - 1]) <= (kf_t[lo] - u))) best = lo - 1;
    return best;
}

// pass 1: decide every event once, remember the decision in a 16-bit tag (0 = no residual, else spline<<8 | circle+1)
// (ncu, profiles/r1e: the 36 FP64 distance evaluations were 71 % of this kernel's instructions, issue-bound at 72 % — hence the
//  FP32 preselection with sortable keys in assoc_one; an earlier shared-memory variant of the FP64 loop had measured slower)
__global__ void __launch_bounds__(AS_THREADS) k_assoc_count(const AssocArgs a, uint16_t *__restrict__ tag,
                                                           uint32_t *__restrict__ block_cnt) {
    __shared__ uint32_t ws[33];
    const int64_t i = (int64_t) blockIdx.x * AS_THREADS + threadIdx.x;
    int s = 0;
    const int bi = i < a.n_ev ? assoc_one(a, i, &s) : -1;
    if (i < a.n_ev) tag[i] = bi >= 0 ? (uint16_t) ((s << 8) | (bi + 1)) : (uint16_t) 0;
    uint32_t tot;
    block_excl_scan(bi >= 0 ? 1u : 0u, ws, &tot);
    if (threadIdx.x == 0) block_cnt[blockIdx.x] = tot;
}

__global__ void k_scan_blocks(uint32_t *cnt, int n, int64_t *off, int64_t *total) {  // single block: one segment per thread
    __shared__ uint32_t ws[33];
    const int per = (n + (int) blockDim.x - 1) / (int) blockDim.x;
    const int b = min(n, (int) threadIdx.x * per), e = min(n, b + per);
    uint32_t sum = 0;
    for (int i = b; i < e; ++i) sum += cnt[i];
    uint32_t tot;
    int64_t run = block_excl_scan(sum, ws, &tot);  // the per-launch total (tagged events) fits 32 bits: n_events < 2^32
    for (int i = b; i < e; ++i) {
        off[i] = run;
        run += cnt[i];
    }
    if (threadIdx.x == 0) *total = tot;
}

// pass 2: ordered compaction of the tagged events into residual records (pure streaming)
__global__ void __launch_bounds__(AS_THREADS) k_assoc_write(const AssocArgs a, const uint16_t *__restrict__ tag,
                                                           const int64_t *__restrict__ block_off,
                                                           double *__restrict__ obs, double *__restrict__ lm,
                                                           double *__restrict__ tt, int *__restrict__ spl,
                                                           int64_t *__restrict__ sel_event, int *__restrict__ sel_circle) {
    __shared__ uint32_t ws[33];
    const int64_t i = (int64_t) blockIdx.x * AS_THREADS + threadIdx.x;
    const uint32_t tg = i < a.n_ev ? tag[i] : 0u;
    uint32_t tot;
    const uint32_t ex = block_excl_scan(tg ? 1u : 0u, ws, &tot);
    if (tg) {
        const int bi = (int) (tg & 0xFF) - 1, s = (int) (tg >> 8);
        const int64_t k = block_off[blockIdx.x] + ex;
        const uint32_t e = a.ev_xyp[i];
        reinterpret_cast<double2 *>(obs)[k] = make_double2((double) ECB_PIX_X(e), (double) ECB_PIX_Y(e));
        const double u = a.ev_t[i];
        sel_event[k] = i;
        sel_circle[k] = bi;  // the evaluation kernels read the landmark from lm_tab[circle]
        if (!a.basis) {      // unfused path: k_prepare needs time and spline, the kernels the explicit landmark
            lm[3 * k] = a.lm_tab[3 * bi];
            lm[3 * k + 1] = a.lm_tab[3 * bi + 1];
            lm[3 * k + 2] = a.lm_tab[3 * bi + 2];
            tt[k] = u;
            spl[k] = s;
        }
        if (a.basis) {  // what k_prepare would compute (findSpan / dersBasisFuns, EventCalibSpline.cpp:173-179)
            const double *kn = a.knots + a.knot_off[s];
            const int sp = find_span_guess(kn, a.ncp[s] + 4, u);
            double N[4];
            basis_dev(kn, sp, u, N);
            reinterpret_cast<double4 *>(a.basis)[k] = make_double4(N[0], N[1], N[2], N[3]);
            a.cp0[k] = a.cp_off[s] + sp - 3;
            a.span[k] = a.span_off[s] + sp - 3;
        }
    }
}

// ------------------------------------------------------------------------------ re-association ----
// k_reassoc_count  pass 1 of the association through the calibrated model: a candidate event (segment, valid pixel, near its
//                  key frame) gets its pose on the spline, its board point X_w, the landmark nearest to X_w and the event-to-rim
//                  error e of that pair; the 16-bit tag of k_assoc_count records the kept ones, so k_scan_blocks and k_assoc_write
//                  write the records as for an association.  A kept event is looked up in the previous records (ordered by
//                  event) for the counts against them, summed with integer atomics.
struct ReassocArgs {
    AssocArgs as;                // events, segments, the association's stamps / window / landmarks
    double max_dt;               // > 0: |t - t_kf| <= max_dt instead of the association's window
    const double *params;        // intr 9 | rot 4C | trans 3C
    int total_cp;
    EcbFold fold;
    double radius, gate_px;
    const int64_t *prev_event;   // the records before the call
    const int *prev_circle;
    int64_t n_prev;
    unsigned long long *counts;  // same, changed, new
};

constexpr int RA_MAX_CIRC = 256;  // > the association's limit of 254 circles

// circle of one candidate event (or -1); L32: FP32 landmarks, lmax: their largest |coordinate|
template <int SO3>
__device__ __forceinline__ int reassoc_one(const ReassocArgs &r, const float4 *L32, float lmax, int64_t i, int *spline_out) {
    const AssocArgs &a = r.as;
    const double u = a.ev_t[i];
    const int s = segment_of(a, u);
    if (s < 0) return -1;
    *spline_out = s;
    const double dt = u - a.kf_t[nearest_kf(a.kf_t, a.K, u)];
    if (r.max_dt > 0.0 ? !(fabs(dt) <= r.max_dt) : !(__dmul_rn(dt, dt) < a.gate2)) return -1;
    const uint32_t e = a.ev_xyp[i];
    if (e & ECB_PIX_INVALID) return -1;
    const double ou = (double) ECB_PIX_X(e), ov = (double) ECB_PIX_Y(e);
    // the pose as the record's evaluation sees it: the basis of k_assoc_write, ecb_pose_eval as in the reprojection metric
    const double *kn = a.knots + a.knot_off[s];
    const int sp = find_span_guess(kn, a.ncp[s] + 4, u);
    double N[4], q[4], t[3], X[3];
    basis_dev(kn, sp, u, N);
    const int c0 = a.cp_off[s] + sp - 3;
    const double *intr = r.params;
    ecb_pose_eval(intr + 9 + 4 * (size_t) c0, intr + 9 + 4 * (size_t) r.total_cp + 3 * (size_t) c0, N, SO3, q, t);
    ecb_board_point(intr, q, t, ou, ov, X);
    if (!(fabs(X[0]) < INFINITY && fabs(X[1]) < INFINITY && fabs(X[2]) < INFINITY)) return -1;
    // Nearest landmark, assoc_one's scheme: FP32 preselection with sortable keys (distance bits | index), the two smallest kept.
    // The FP32 distance of any landmark is within 1e-6 S of the exact one (S: the largest |coordinate| of X_w and the landmarks),
    // so when the runner-up's lower bound clears the winner's upper bound by 1e-5 S the winner is the exact FP64 arg-min; else
    // the exact FP64 loop decides (ties -> the smaller index).
    int bi = -1;
    {
        const float xf = (float) X[0], yf = (float) X[1], zf = (float) X[2];
        uint32_t k1 = 0xFFFFFFFFu, k2 = 0xFFFFFFFFu;
#pragma unroll 1  // unrolled by 4, the quaternion variant spills 8 bytes
        for (int c = 0; c < a.n_circ; ++c) {
            const float4 L = L32[c];
            const float dx = xf - L.x, dy = yf - L.y, dz = zf - L.z;
            const uint32_t k = (__float_as_uint(fmaf(dx, dx, fmaf(dy, dy, dz * dz))) & 0xFFFFFF00u) | (uint32_t) c;
            k2 = min(k2, max(k, k1));
            k1 = min(k1, k);
        }
        const float d1 = sqrtf(__uint_as_float(k1 | 0xFFu)), d2 = sqrtf(__uint_as_float(k2 & 0xFFFFFF00u));
        const float S = fmaxf(lmax, fmaxf(fabsf(xf), fmaxf(fabsf(yf), fabsf(zf))));
        if (d2 > d1 * 1.0001f + 1e-5f * S) {  // NaN (one circle, overflow): the FP64 loop
            bi = (int) (k1 & 0xFFu);
        } else {
            double bd = 0.0;
            for (int c = 0; c < a.n_circ; ++c) {
                const double *L = a.lm_tab + 3 * c;
                const double dx = X[0] - L[0], dy = X[1] - L[1], dz = X[2] - L[2];
                const double dd = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
                if (bi < 0 || dd < bd) {
                    bi = c;
                    bd = dd;
                }
            }
        }
    }
    const double *L = a.lm_tab + 3 * bi;
    const double err = ecb_rim_reprojection(intr, r.fold, q, t, ou, ov, L[0], L[1], L[2], r.radius);
    return fabs(err) < r.gate_px ? bi : -1;  // NaN: not kept
}

template <int SO3>
__global__ void __launch_bounds__(AS_THREADS) k_reassoc_count(const ReassocArgs r, uint16_t *__restrict__ tag,
                                                             uint32_t *__restrict__ block_cnt) {
    __shared__ uint32_t ws[33];
    __shared__ float4 L32[RA_MAX_CIRC];
    __shared__ uint32_t lmax_bits;  // a non-negative float: its bits order as the values (integer max: deterministic)
    const AssocArgs &a = r.as;
    if (threadIdx.x == 0) lmax_bits = 0;
    __syncthreads();
    for (int c = threadIdx.x; c < a.n_circ; c += AS_THREADS) {
        const double *L = a.lm_tab + 3 * c;
        const float4 v = make_float4((float) L[0], (float) L[1], (float) L[2], 0.f);
        L32[c] = v;
        atomicMax(&lmax_bits, __float_as_uint(fmaxf(fabsf(v.x), fmaxf(fabsf(v.y), fabsf(v.z)))));
    }
    __syncthreads();
    const int64_t i = (int64_t) blockIdx.x * AS_THREADS + threadIdx.x;
    int s = 0;
    const int bi = i < a.n_ev ? reassoc_one<SO3>(r, L32, __uint_as_float(lmax_bits), i, &s) : -1;
    if (i < a.n_ev) tag[i] = bi >= 0 ? (uint16_t) ((s << 8) | (bi + 1)) : (uint16_t) 0;
    uint32_t tot;
    block_excl_scan(bi >= 0 ? 1u : 0u, ws, &tot);
    if (threadIdx.x == 0) block_cnt[blockIdx.x] = tot;
    uint32_t same = 0, changed = 0, fresh = 0;
    if (bi >= 0) {
        int64_t lo = 0, hi = r.n_prev;  // lower_bound of i in the previous records' events
        while (lo < hi) {
            const int64_t m = (lo + hi) >> 1;
            if (r.prev_event[m] < i) lo = m + 1; else hi = m;
        }
        if (lo < r.n_prev && r.prev_event[lo] == i) {
            same = r.prev_circle[lo] == bi;
            changed = !same;
        } else {
            fresh = 1;
        }
    }
    same = __reduce_add_sync(0xffffffffu, same);
    changed = __reduce_add_sync(0xffffffffu, changed);
    fresh = __reduce_add_sync(0xffffffffu, fresh);
    if ((threadIdx.x & 31) == 0) {
        if (same) atomicAdd(&r.counts[0], (unsigned long long) same);
        if (changed) atomicAdd(&r.counts[1], (unsigned long long) changed);
        if (fresh) atomicAdd(&r.counts[2], (unsigned long long) fresh);
    }
}

// ------------------------------------------------------------------- residual and reprojection reports ----
// Both reports evaluate one value per record (a metric) and the same statistics per group:
// k_record_report  the loads of k_cost and the metric of record k -> out[k]; optional count of the NaN values (integer atomics,
//                  one per warp)
// k_group_keys     group of every record (key) and its index; a stable radix sort of (key, index) keeps record order per group
// k_group_start    lower bounds of every group in the sorted keys (as k_span_start)
// k_group_stats    one block per group, fixed shape: thread-strided partials in record order, then a shared-memory tree
constexpr int RG_THREADS = 256;

// (s, c) += v with the rounding error of s + v kept in c (Neumaier); Knuth's TwoSum, exact without branches
ECB_HD void ecb_comp_add(double &s, double &c, double v) {
    const double t = s + v, bp = t - s;
    c += (s - (t - bp)) + (v - bp);
    s = t;
}

// The statistics of one group: add() one record's value, merge() another partial, result() the group.  Host and device: the
// total over the groups is the tree's merge.
struct ResidualStats {  // raw residuals r (board units)
    using Group = ecb_residual_group;
    Group q;
    double huber;
    ECB_HD void add(double v) {
        // the Huber expressions of ecb_residual.h: rho = r^2 inside the band, 2 delta |r| - delta^2 outside
        const double a2 = huber * huber, s2 = v * v;
        double rho = s2;
        if (s2 > a2) {
            rho = 2.0 * huber * fabs(v) - a2;
            ++q.n_downweighted;
        }
        ++q.count;
        q.sum += v;
        q.sum_sq += s2;
        q.max_abs = fmax(q.max_abs, fabs(v));
        q.cost += 0.5 * rho;
    }
    ECB_HD void merge(const ResidualStats &o) {
        q.count += o.q.count;
        q.n_downweighted += o.q.n_downweighted;
        q.sum += o.q.sum;
        q.sum_sq += o.q.sum_sq;
        q.max_abs = fmax(q.max_abs, o.q.max_abs);
        q.cost += o.q.cost;
    }
    ECB_HD Group result() const { return q; }
};

// Reprojection errors e (pixels): valid records counted and summed, NaN ones counted in n_invalid only.  e is signed and its
// sums cancel (the mean error of a group is near 0 when the fit is good), so sum e is compensated (Neumaier per thread, TwoSum
// in the tree): it keeps the relative accuracy of the sum itself instead of n eps sum |e|.
struct ReprojectionStats {
    using Group = ecb_reprojection_group;
    Group q;
    double comp;  // rounding error of q.sum
    ECB_HD void add(double v) {
        if (isnan(v)) {
            ++q.n_invalid;
            return;
        }
        ++q.count;
        ecb_comp_add(q.sum, comp, v);
        q.sum_sq += v * v;
        q.max_abs = fmax(q.max_abs, fabs(v));
    }
    ECB_HD void merge(const ReprojectionStats &o) {
        q.count += o.q.count;
        q.n_invalid += o.q.n_invalid;
        comp += o.comp;
        ecb_comp_add(q.sum, comp, o.q.sum);
        q.sum_sq += o.q.sum_sq;
        q.max_abs = fmax(q.max_abs, o.q.max_abs);
    }
    ECB_HD Group result() const {
        Group g = q;
        g.sum = q.sum + comp;
        return g;
    }
};

// The metrics: at() takes them from the context and the host intrinsics, stats() starts a group of their statistics.
struct ResidualMetric {  // r_k = ||X_w - L|| - radius, the raw residual of ecb_residual (board units)
    using Stats = ResidualStats;
    static constexpr const char *report = "residual";
    double radius, huber;
    static ResidualMetric at(const CostState *st, const double *) { return {st->radius, st->huber}; }
    Stats stats() const { return Stats{{}, huber}; }
    template <int SO3>
    __device__ __forceinline__ double operator()(const double *intr, const double *rot, const double *trans, const double b[4],
                                                 double2 o, const double L[3]) const {
        return SO3 ? ecb_residual_so3<false>(intr, rot, trans, b, o.x, o.y, L[0], L[1], L[2], radius, huber, nullptr).raw
                   : ecb_residual<false>(intr, rot, trans, b, o.x, o.y, L[0], L[1], L[2], radius, huber, nullptr).raw;
    }
};

struct RimReprojectionMetric {  // e_k in pixels: the record's pose (ecb_pose_eval), then ecb_rim_reprojection; NaN when not projectable
    using Stats = ReprojectionStats;
    static constexpr const char *report = "reprojection";
    double radius;
    EcbFold fold;
    static RimReprojectionMetric at(const CostState *st, const double *intr) { return {st->radius, ecb_inverse_radial_fold_host(intr + 4)}; }
    Stats stats() const { return Stats{{}, 0.0}; }
    template <int SO3>
    __device__ __forceinline__ double operator()(const double *intr, const double *rot, const double *trans, const double b[4],
                                                 double2 o, const double L[3]) const {
        double q[4], t[3];
        ecb_pose_eval(rot, trans, b, SO3, q, t);
        return ecb_rim_reprojection(intr, fold, q, t, o.x, o.y, L[0], L[1], L[2], radius);
    }
};

template <int SO3, class Metric>
__global__ void __launch_bounds__(256) k_record_report(const double *__restrict__ obs, const double *__restrict__ lm,
                                                       const int *__restrict__ circ, const double *__restrict__ lm_tab,
                                                       const double *__restrict__ basis, const int *__restrict__ cp0, int64_t n,
                                                       const double *__restrict__ params, int total_cp, const Metric m,
                                                       double *__restrict__ out, unsigned long long *__restrict__ n_invalid) {
    const double *intr = params, *rot = params + 9, *trans = params + 9 + 4 * (size_t) total_cp;
    const RecordView rv{obs, lm, circ, lm_tab, basis, cp0};
    unsigned bad = 0;
    for (int64_t k = (int64_t) blockIdx.x * 256 + threadIdx.x; k < n; k += (int64_t) gridDim.x * 256) {
        int c0;
        double b[4], L[3];
        double2 o;
        rv.load(k, c0, b, o, L);
        const double v = m.template operator()<SO3>(intr, rot + 4 * (size_t) c0, trans + 3 * (size_t) c0, b, o, L);
        out[k] = v;
        bad += isnan(v) ? 1u : 0u;
    }
    if (n_invalid) {
        bad = __reduce_add_sync(0xffffffffu, bad);
        if ((threadIdx.x & 31) == 0 && bad) atomicAdd(n_invalid, (unsigned long long) bad);
    }
}

struct GroupKeyArgs {
    int by;                    // ECB_RESIDUALS_BY_*
    const int64_t *sel_event;  // association: event of record k
    const int *sel_circle;     // association: circle of record k
    const double *ev_t, *kf_t;
    int K;
    const double *obs;
    int width, height, cell, ncx;
    uint32_t outside;          // key of the records that count in the total only (= number of groups)
};

__global__ void k_group_keys(const GroupKeyArgs a, int64_t n, uint64_t *__restrict__ key, uint32_t *__restrict__ idx) {
    for (int64_t k = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t) gridDim.x * blockDim.x) {
        uint32_t g;
        if (a.by == ECB_RESIDUALS_BY_KEYFRAME) {
            g = (uint32_t) nearest_kf(a.kf_t, a.K, a.ev_t[a.sel_event[k]]);
        } else if (a.by == ECB_RESIDUALS_BY_CIRCLE) {
            g = (uint32_t) a.sel_circle[k];
        } else {
            const double2 o = reinterpret_cast<const double2 *>(a.obs)[k];
            if (o.x >= 0.0 && o.x < (double) a.width && o.y >= 0.0 && o.y < (double) a.height)
                g = (uint32_t) floor(o.y / a.cell) * (uint32_t) a.ncx + (uint32_t) floor(o.x / a.cell);
            else
                g = a.outside;  // also NaN
        }
        key[k] = g;
        idx[k] = (uint32_t) k;
    }
}

// start[g] = first sorted position with key >= g, g = 0 .. n_keys (start[n_keys] = n)
__global__ void k_group_start(const uint64_t *__restrict__ skey, int64_t n, int n_keys, int64_t *__restrict__ start) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g > n_keys) return;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t m = (lo + hi) >> 1;
        if (skey[m] < (uint64_t) g) lo = m + 1; else hi = m;
    }
    start[g] = lo;
}

// s: an empty group of the statistics (carrying their parameters)
template <class Stats>
__global__ void __launch_bounds__(RG_THREADS) k_group_stats(const double *__restrict__ v, const uint32_t *__restrict__ sidx,
                                                            const int64_t *__restrict__ start, Stats s,
                                                            typename Stats::Group *__restrict__ out) {
    __shared__ Stats sh[RG_THREADS];
    const int g = blockIdx.x, t = threadIdx.x;
    const int64_t b = start[g], e = start[g + 1];
    for (int64_t i = b + t; i < e; i += RG_THREADS) s.add(v[sidx[i]]);
    sh[t] = s;
    __syncthreads();
    for (int o = RG_THREADS / 2; o > 0; o >>= 1) {
        if (t < o) sh[t].merge(sh[t + o]);
        __syncthreads();
    }
    if (t == 0) out[g] = sh[0].result();
}

// ------------------------------------------------------------------------ outlier rejection ----
// k_reject_count  keep flag of every record (|r_k| <= threshold, and its key frame not dropped) and the per-block count
// k_reject_write  ordered compaction of the kept records into the spare buffers (k_assoc_write's scheme; blocks overlap, so
//                 not in place)
struct RejectArgs {
    const double *r;           // r_k (k_record_report)
    double max_abs;
    const uint8_t *drop;       // per key frame, or null
    const double *kf_t;        // the association's stamps (drop != null)
    int K;
    const int64_t *sel_event;  // association: event of record k
    const double *ev_t;
    int64_t n;
};

__global__ void __launch_bounds__(AS_THREADS) k_reject_count(const RejectArgs a, uint8_t *__restrict__ keep,
                                                            uint32_t *__restrict__ block_cnt) {
    __shared__ uint32_t ws[33];
    const int64_t k = (int64_t) blockIdx.x * AS_THREADS + threadIdx.x;
    uint32_t kp = 0;
    if (k < a.n) {
        kp = fabs(a.r[k]) <= a.max_abs ? 1u : 0u;  // NaN: removed
        if (kp && a.drop && a.drop[nearest_kf(a.kf_t, a.K, a.ev_t[a.sel_event[k]])]) kp = 0;
        keep[k] = (uint8_t) kp;
    }
    uint32_t tot;
    block_excl_scan(kp, ws, &tot);
    if (threadIdx.x == 0) block_cnt[blockIdx.x] = tot;
}

// the record arrays of one buffer set; a null pointer is an array the path does not hold
struct RecordPtrs {
    double2 *obs;
    double4 *basis;
    int *cp0, *span;
    int64_t *sel_event;
    int *sel_circle;
    double *lm, *tt;
    int *spl;
};

__global__ void __launch_bounds__(AS_THREADS) k_reject_write(const uint8_t *__restrict__ keep, const int64_t *__restrict__ block_off,
                                                            int64_t n, const RecordPtrs s, const RecordPtrs d) {
    __shared__ uint32_t ws[33];
    const int64_t k = (int64_t) blockIdx.x * AS_THREADS + threadIdx.x;
    const uint32_t kp = k < n ? keep[k] : 0u;
    uint32_t tot;
    const uint32_t ex = block_excl_scan(kp, ws, &tot);
    if (!kp) return;
    const int64_t o = block_off[blockIdx.x] + ex;
    d.obs[o] = s.obs[k];
    d.basis[o] = s.basis[k];
    d.cp0[o] = s.cp0[k];
    d.span[o] = s.span[k];
    if (s.sel_event) {
        d.sel_event[o] = s.sel_event[k];
        d.sel_circle[o] = s.sel_circle[k];
    }
    if (s.lm) {
        d.lm[3 * o] = s.lm[3 * k];
        d.lm[3 * o + 1] = s.lm[3 * k + 1];
        d.lm[3 * o + 2] = s.lm[3 * k + 2];
        d.tt[o] = s.tt[k];
        d.spl[o] = s.spl[k];
    }
}

// ------------------------------------------------------------------------ key-frame reprojection ----
// k_keyframe_reproj one thread per (key frame, circle): the board point at the key frame's pose, projected
// kf_t[K], circ[K][nc][3] (cx cy r), lm[nc][3] -> proj[K][nc][2], err[K][nc]; the segment and span lookup of k_pose_cov
template <int SO3>
__global__ void __launch_bounds__(128) k_keyframe_reproj(const double *__restrict__ kf_t, const double *__restrict__ circ,
                                                         const double *__restrict__ lm, int K, int nc, EcbSplineView sv,
                                                         const double *__restrict__ params, EcbFold fold,
                                                         double *__restrict__ proj, double *__restrict__ err) {
    const int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t) K * nc) return;
    const int kf = (int) (i / nc), c = (int) (i % nc);
    const double *ci = circ + 3 * i;
    double pu = NAN, pv = NAN, e = NAN;
    const double u = kf_t[kf];
    const double *kn = nullptr;
    int nk = 0;
    const int s = sv.segment(u, &kn, &nk);
    if (ci[2] >= 0.0 && s >= 0) {
        const int span = find_span_dev(kn, nk, u);
        double N[4], q[4], t[3];
        basis_dev(kn, span, u, N);
        const int c0 = sv.cp_off[s] + span - 3;
        ecb_pose_eval(params + 9 + 4 * (size_t) c0, params + 9 + 4 * (size_t) sv.total_cp + 3 * (size_t) c0, N, SO3, q, t);
        const double P[3] = {lm[3 * c] - t[0], lm[3 * c + 1] - t[1], lm[3 * c + 2] - t[2]};
        double pc[3], a, b;
        ecb_quat_rotate(q, P, true, pc);
        if (ecb_project(params, fold, pc, a, b)) {
            const double d = sqrt((a - ci[0]) * (a - ci[0]) + (b - ci[1]) * (b - ci[1]));
            if (d < INFINITY) {
                pu = a;
                pv = b;
                e = d;
            }
        }
    }
    proj[2 * i] = pu;
    proj[2 * i + 1] = pv;
    err[i] = e;
}

int prepare_records(ecb_ctx *ctx, CostState *st, bool have_basis = false) {
    int rc;
    const int64_t n = st->n_res;
    const size_t nn = (size_t) std::max<int64_t>(n, 1);
    if ((rc = ecb_reserve(ctx, st->basis, nn * 32))) return rc;
    if ((rc = ecb_reserve(ctx, st->cp0, nn * 4))) return rc;
    if ((rc = ecb_reserve(ctx, st->span, nn * 4))) return rc;
    if ((rc = ecb_reserve(ctx, st->flags, 16))) return rc;
    if ((rc = ecb_reserve(ctx, st->span_start, (size_t) (st->total_spans + 2) * 8))) return rc;
    ECB_CUDA(ctx, cudaMemsetAsync(st->flags.p, 0, 16, ctx->stream));
    st->h_span_start.assign((size_t) st->total_spans + 1, 0);
    st->n_items = 0;
    if (n == 0) return ECB_OK;
    if (!have_basis)
    k_prepare<<<(unsigned) ((n + 255) / 256), 256, 0, ctx->stream>>>(
        (const double *) st->tt.p, (const int *) st->spl.p, n, (const double *) st->d_knots.p, (const int *) st->d_knot_off.p,
        (const int *) st->d_ncp.p, (const int *) st->d_cp_off.p, (const int *) st->d_span_off.p, (double *) st->basis.p,
        (int *) st->cp0.p, (int *) st->span.p, (uint32_t *) st->flags.p);
    ECB_LAUNCHED(ctx);
    k_span_start<<<(st->total_spans + 1 + 127) / 128, 128, 0, ctx->stream>>>((const int *) st->span.p, n, st->total_spans,
                                                                           (int64_t *) st->span_start.p);
    ECB_LAUNCHED(ctx);
    uint32_t flag = 0;
    ECB_CUDA(ctx, cudaMemcpyAsync((int64_t *) st->span_start.p + st->total_spans + 1, st->flags.p, 4, cudaMemcpyDeviceToDevice,
                                  ctx->stream));  // one staged copy for both
    {
        std::vector<int64_t> tmp((size_t) st->total_spans + 2);
        if ((rc = ecb_d2h(ctx, tmp.data(), st->span_start.p, tmp.size() * 8))) return rc;
        std::copy(tmp.begin(), tmp.begin() + st->total_spans + 1, st->h_span_start.begin());
        flag = (uint32_t) (tmp[(size_t) st->total_spans + 1] & 0xFFFFFFFF);
    }
    if (flag & 1u) return ecb_fail(ctx, ECB_ERR_ARG, "a residual's time stamp lies outside its spline's knot range");
    if (flag & 2u) return ecb_fail(ctx, ECB_ERR_ARG, "residual records must be ordered by (spline, time)");
    // work items: chunks of <= chunk residuals inside one span (a function of the record counts and the SM count only =>
    // deterministic reduction order).  One item is one warp's latency-bound pass (0.45 ms per 2048 residuals on B200), so the
    // chunk is sized to hand every resident warp of k_normal_eq the same number of items: small residual sets (a time slice
    // of the end-to-end pipeline, one rank of eight) then use all warps with shorter items instead of half of them.
    int chunk = CHUNK;
    {
        const int64_t warps = (int64_t) ctx->sm_count * (st->so3 ? 1 : 2) * NE_WARPS;
        int64_t rounds = std::max<int64_t>(1, (n + warps * CHUNK - 1) / (warps * CHUNK));
        chunk = (int) (((n + warps * rounds - 1) / (warps * rounds) + 31) / 32 * 32);
        chunk = std::min(std::max(chunk, 256), CHUNK);
        static const int chunk_cap = getenv("ECB_NE_CHUNK") ? atoi(getenv("ECB_NE_CHUNK")) : 1536;  // shorter items: no partial last round (1.86 -> 1.81 ms)
        if (chunk_cap >= 256 && chunk > chunk_cap) {
            rounds = std::max<int64_t>(1, (n + warps * chunk_cap - 1) / (warps * chunk_cap));
            chunk = std::min((int) (((n + warps * rounds - 1) / (warps * rounds) + 31) / 32 * 32), chunk_cap);
        }
        for (; chunk < CHUNK; chunk += 32) {  // the partial chunks at span ends add items: grow until the count fits
            int64_t cnt = 0;
            for (int s = 0; s < st->total_spans; ++s)
                cnt += (st->h_span_start[(size_t) s + 1] - st->h_span_start[(size_t) s] + chunk - 1) / chunk;
            if (cnt <= warps * rounds) break;
        }
    }
    std::vector<Item> items;
    std::vector<int> item_start((size_t) st->total_spans + 1, 0);
    for (int s = 0; s < st->total_spans; ++s) {
        item_start[(size_t) s] = (int) items.size();
        for (int64_t b = st->h_span_start[(size_t) s]; b < st->h_span_start[(size_t) s + 1]; b += chunk)
            items.push_back(Item{b, std::min<int64_t>(b + chunk, st->h_span_start[(size_t) s + 1]), s, 0});
    }
    item_start[(size_t) st->total_spans] = (int) items.size();
    st->n_items = (int) items.size();
    const size_t ni = std::max<size_t>(items.size(), 1);
    if ((rc = ecb_reserve(ctx, st->items, ni * sizeof(Item) + item_start.size() * 4 + 64))) return rc;
    if ((rc = ecb_reserve(ctx, st->part, ni * PART_STRIDE * 8))) return rc;
    if ((rc = ecb_reserve(ctx, st->out, ((size_t) st->total_spans * OUT_STRIDE + 8) * 8))) return rc;
    if ((rc = ecb_reserve(ctx, st->cost_part, 4096 * 8))) return rc;
    if (!items.empty())
        if ((rc = ecb_h2d(ctx, st->items.p, items.data(), items.size() * sizeof(Item)))) return rc;
    return ecb_h2d(ctx, (char *) st->items.p + ni * sizeof(Item), item_start.data(), item_start.size() * 4);  // staged: no sync needed
}

int upload_params(ecb_ctx *ctx, CostState *st, const double *intr, const double *rot, const double *trans) {
    int rc;
    const size_t C = (size_t) st->total_cp;
    if ((rc = ecb_reserve(ctx, st->params, (9 + 7 * C) * 8))) return rc;
    double *p = (double *) st->params.p;
    if ((rc = ecb_h2d(ctx, p, intr, 72))) return rc;
    if ((rc = ecb_h2d(ctx, p + 9, rot, 32 * C))) return rc;
    return ecb_h2d(ctx, p + 9 + 4 * C, trans, 24 * C);
}

}  // namespace

extern "C" {

void ecb_cost_free(ecb_ctx *ctx) {
    if (!ctx || !ctx->cost) return;
    CostState *st = (CostState *) ctx->cost;
    DevBuf *bufs[] = {&st->d_knots, &st->d_knot_off, &st->d_ncp, &st->d_cp_off, &st->d_span_off, &st->obs, &st->lm, &st->tt,
                      &st->spl, &st->basis, &st->cp0, &st->span, &st->span_start, &st->items, &st->part, &st->out, &st->params,
                      &st->cost_part, &st->flags, &st->ev_flag, &st->ev_cnt, &st->ev_tag, &st->kf_t, &st->kf_circ, &st->kf_c32, &st->lm_tab,
                      &st->sel_event, &st->sel_circle, &st->rep_r, &st->rep_key[0], &st->rep_key[1], &st->rep_idx[0],
                      &st->rep_idx[1], &st->rep_hist, &st->rep_start, &st->rep_out, &st->rep_kf, &st->rep_io};
    for (DevBuf *b : bufs)
        if (b->p) cudaFree(b->p);
    for (DevBuf &b : st->rej)
        if (b.p) cudaFree(b.p);
    delete st;
    ctx->cost = nullptr;
}

int ecb_cost_setup(ecb_ctx *ctx, int n_splines, const int32_t *n_cp, const double *knots, double circle_radius,
                   double huber_delta) {
    if (!ctx || n_splines < 1 || !n_cp || !knots) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    CostState *st = state(ctx);
    st->n_splines = n_splines;
    st->n_cp.assign(n_cp, n_cp + n_splines);
    st->cp_off.clear();
    st->span_off.clear();
    st->knot_off.clear();
    int co = 0, so = 0, ko = 0;
    for (int s = 0; s < n_splines; ++s) {
        if (n_cp[s] < 4) return ecb_fail(ctx, ECB_ERR_ARG, "spline %d has %d control points (< degree + 1)", s, n_cp[s]);
        st->cp_off.push_back(co);
        st->span_off.push_back(so);
        st->knot_off.push_back(ko);
        co += n_cp[s];
        so += n_cp[s] - 3;
        ko += n_cp[s] + 4;
    }
    st->total_cp = co;
    st->total_spans = so;
    st->knots.assign(knots, knots + ko);
    ++ctx->spline_gen;
    st->radius = circle_radius;
    st->huber = huber_delta;
    st->n_res = 0;
    st->n_items = 0;
    st->assoc = false;
    int rc;
    if ((rc = ecb_reserve(ctx, st->d_knots, (size_t) ko * 8))) return rc;
    if ((rc = ecb_reserve(ctx, st->d_knot_off, (size_t) n_splines * 4))) return rc;
    if ((rc = ecb_reserve(ctx, st->d_ncp, (size_t) n_splines * 4))) return rc;
    if ((rc = ecb_reserve(ctx, st->d_cp_off, (size_t) n_splines * 4))) return rc;
    if ((rc = ecb_reserve(ctx, st->d_span_off, (size_t) n_splines * 4))) return rc;
    ECB_CUDA(ctx, cudaMemcpyAsync(st->d_knots.p, knots, (size_t) ko * 8, cudaMemcpyHostToDevice, ctx->stream));
    ECB_CUDA(ctx, cudaMemcpyAsync(st->d_knot_off.p, st->knot_off.data(), (size_t) n_splines * 4, cudaMemcpyHostToDevice, ctx->stream));
    ECB_CUDA(ctx, cudaMemcpyAsync(st->d_ncp.p, st->n_cp.data(), (size_t) n_splines * 4, cudaMemcpyHostToDevice, ctx->stream));
    ECB_CUDA(ctx, cudaMemcpyAsync(st->d_cp_off.p, st->cp_off.data(), (size_t) n_splines * 4, cudaMemcpyHostToDevice, ctx->stream));
    ECB_CUDA(ctx, cudaMemcpyAsync(st->d_span_off.p, st->span_off.data(), (size_t) n_splines * 4, cudaMemcpyHostToDevice, ctx->stream));
    return ecb_check(ctx, ecb_stream_sync(ctx), "cost setup");
}

int ecb_cost_set_rotation_model(ecb_ctx *ctx, int use_so3) {
    if (!ctx || !ctx->cost) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_cost_setup first");
    if (use_so3 != 0 && use_so3 != 1) return ECB_ERR_ARG;
    ((CostState *) ctx->cost)->so3 = use_so3;
    ++ctx->spline_gen;
    return ECB_OK;
}

int ecb_cost_set_constant_intrinsics(ecb_ctx *ctx, uint32_t mask) {
    if (!ctx) return ECB_ERR_ARG;
    if (mask > ECB_ALL_INTRINSICS) return ecb_fail(ctx, ECB_ERR_ARG, "constant intrinsics mask 0x%x has bits above the 9 intrinsics", mask);
    if (mask != ctx->const_intrinsics) {
        ctx->const_intrinsics = mask;
        ++ctx->spline_gen;  // Z depends on the free parameters: a covariance computed before no longer answers ecb_pose_covariance
    }
    return ECB_OK;
}

int ecb_cost_spline_view(ecb_ctx *ctx, EcbSplineView *v) {
    if (!ctx || !ctx->cost) return ECB_ERR_STATE;
    const CostState *st = (const CostState *) ctx->cost;
    v->knots = (const double *) st->d_knots.p;
    v->knot_off = (const int *) st->d_knot_off.p;
    v->ncp = (const int *) st->d_ncp.p;
    v->cp_off = (const int *) st->d_cp_off.p;
    v->n_splines = st->n_splines;
    v->total_cp = st->total_cp;
    v->so3 = st->so3;
    return ECB_OK;
}

int ecb_cost_layout(ecb_ctx *ctx, int32_t *total_cp, int32_t *total_spans, int64_t *n_residuals, int64_t *out_doubles) {
    if (!ctx || !ctx->cost) return ECB_ERR_STATE;
    CostState *st = (CostState *) ctx->cost;
    if (total_cp) *total_cp = st->total_cp;
    if (total_spans) *total_spans = st->total_spans;
    if (n_residuals) *n_residuals = st->n_res;
    if (out_doubles) *out_doubles = (int64_t) st->total_spans * OUT_STRIDE + 2;
    return ECB_OK;
}

int ecb_cost_set_residuals(ecb_ctx *ctx, const double *obs_xy, const double *lm_xyz, const double *t, const int32_t *spline,
                           int64_t n) {
    if (!ctx || !ctx->cost) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_cost_setup first");
    if (n < 0 || (n > 0 && (!obs_xy || !lm_xyz || !t || !spline))) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    CostState *st = (CostState *) ctx->cost;
    int rc;
    const size_t nn = (size_t) std::max<int64_t>(n, 1);
    if ((rc = ecb_reserve(ctx, st->obs, nn * 16))) return rc;
    if ((rc = ecb_reserve(ctx, st->lm, nn * 24))) return rc;
    if ((rc = ecb_reserve(ctx, st->tt, nn * 8))) return rc;
    if ((rc = ecb_reserve(ctx, st->spl, nn * 4))) return rc;
    if (n > 0) {
        ECB_CUDA(ctx, cudaMemcpyAsync(st->obs.p, obs_xy, (size_t) n * 16, cudaMemcpyHostToDevice, ctx->stream));
        ECB_CUDA(ctx, cudaMemcpyAsync(st->lm.p, lm_xyz, (size_t) n * 24, cudaMemcpyHostToDevice, ctx->stream));
        ECB_CUDA(ctx, cudaMemcpyAsync(st->tt.p, t, (size_t) n * 8, cudaMemcpyHostToDevice, ctx->stream));
        ECB_CUDA(ctx, cudaMemcpyAsync(st->spl.p, spline, (size_t) n * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    st->n_res = n;
    st->use_circ = false;
    st->assoc = false;
    return prepare_records(ctx, st);
}

// pass 2 of an association from the tags in st->ev_tag and the block offsets in st->ev_flag: the record buffers sized for
// `total`, then k_assoc_write (fused: the basis pass folded in); async
static int write_assoc_records(ecb_ctx *ctx, CostState *st, AssocArgs a, int nb, int64_t total, bool fused) {
    int rc;
    const size_t nn = (size_t) std::max<int64_t>(total, 1);
    if ((rc = ecb_reserve(ctx, st->obs, nn * 16))) return rc;
    if ((rc = ecb_reserve(ctx, st->lm, nn * 24))) return rc;
    if ((rc = ecb_reserve(ctx, st->tt, nn * 8))) return rc;
    if ((rc = ecb_reserve(ctx, st->spl, nn * 4))) return rc;
    if ((rc = ecb_reserve(ctx, st->sel_event, nn * 8))) return rc;
    if ((rc = ecb_reserve(ctx, st->sel_circle, nn * 4))) return rc;
    a.cp_off = (const int *) st->d_cp_off.p;
    a.span_off = (const int *) st->d_span_off.p;
    a.basis = nullptr;
    a.cp0 = a.span = nullptr;
    if (fused) {
        if ((rc = ecb_reserve(ctx, st->basis, nn * 32))) return rc;
        if ((rc = ecb_reserve(ctx, st->cp0, nn * 4))) return rc;
        if ((rc = ecb_reserve(ctx, st->span, nn * 4))) return rc;
        a.basis = (double *) st->basis.p;
        a.cp0 = (int *) st->cp0.p;
        a.span = (int *) st->span.p;
    }
    k_assoc_write<<<nb, AS_THREADS, 0, ctx->stream>>>(a, (const uint16_t *) st->ev_tag.p, (const int64_t *) st->ev_flag.p, (double *) st->obs.p, (double *) st->lm.p,
                                                      (double *) st->tt.p, (int *) st->spl.p, (int64_t *) st->sel_event.p,
                                                      (int *) st->sel_circle.p);
    ECB_LAUNCHED(ctx);
    return ECB_OK;
}

// the association's arguments for the current events and splines (pass 1 reads cp_off for the fused basis of its records)
static void assoc_args(ecb_ctx *ctx, CostState *st, AssocArgs &a) {
    memset(&a, 0, sizeof a);
    a.ev_t = (const double *) ctx->ev_t.p;
    a.ev_xyp = (const uint32_t *) ctx->ev_xyp.p;
    a.n_ev = ctx->n_events;
    a.knots = (const double *) st->d_knots.p;
    a.knot_off = (const int *) st->d_knot_off.p;
    a.ncp = (const int *) st->d_ncp.p;
    a.n_splines = st->n_splines;
    a.lm_tab = (const double *) st->lm_tab.p;
    a.cp_off = (const int *) st->d_cp_off.p;
}

static int cost_associate(ecb_ctx *ctx, const double *kf_time, const double *kf_circles, int n_keyframes, int n_circles,
                          const double *landmarks_xyz, double motion_time_step, int64_t *n_residuals, bool on_device);

int ecb_cost_associate(ecb_ctx *ctx, const double *kf_time, const double *kf_circles, int n_keyframes, int n_circles,
                       const double *landmarks_xyz, double motion_time_step, int64_t *n_residuals) {
    return cost_associate(ctx, kf_time, kf_circles, n_keyframes, n_circles, landmarks_xyz, motion_time_step, n_residuals, false);
}

int ecb_cost_associate_device(ecb_ctx *ctx, const double *d_kf_time, const double *d_kf_circles, int n_keyframes, int n_circles,
                              const double *d_landmarks_xyz, double motion_time_step, int64_t *n_residuals) {
    return cost_associate(ctx, d_kf_time, d_kf_circles, n_keyframes, n_circles, d_landmarks_xyz, motion_time_step, n_residuals, true);
}

static int cost_associate(ecb_ctx *ctx, const double *kf_time, const double *kf_circles, int n_keyframes, int n_circles,
                          const double *landmarks_xyz, double motion_time_step, int64_t *n_residuals, bool on_device) {
    if (!ctx || !ctx->cost) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_cost_setup first");
    if (!kf_time || !kf_circles || !landmarks_xyz || n_keyframes < 1 || n_circles < 1) return ECB_ERR_ARG;
    if (ctx->n_events <= 0) return ecb_fail(ctx, ECB_ERR_STATE, "no events loaded");
    if (ctx->n_events > 0xFFFFFFFFll) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "association over more than 2^32-1 events per context");
    cudaSetDevice(ctx->device);
    CostState *st = (CostState *) ctx->cost;
    int rc;
    const int64_t n = ctx->n_events;
    const int nb = (int) ((n + AS_THREADS - 1) / AS_THREADS);
    if (!on_device) {
        if ((rc = ecb_reserve(ctx, st->kf_t, (size_t) n_keyframes * 8))) return rc;
        if ((rc = ecb_reserve(ctx, st->kf_circ, (size_t) n_keyframes * n_circles * 24))) return rc;
    }
    if ((rc = ecb_reserve(ctx, st->lm_tab, (size_t) n_circles * 24))) return rc;
    const int n_circ32 = (n_circles + 1) & ~1;
    if ((rc = ecb_reserve(ctx, st->kf_c32, (size_t) n_keyframes * n_circ32 * 8))) return rc;
    if (n_circles > 254 || st->n_splines > 255) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "more than 254 circles or 255 spline segments");
    if ((rc = ecb_reserve(ctx, st->ev_cnt, (size_t) nb * 4 + 16))) return rc;
    if ((rc = ecb_reserve(ctx, st->ev_tag, (size_t) n * 2 + 16))) return rc;
    if ((rc = ecb_reserve(ctx, st->ev_flag, (size_t) nb * 8 + 16))) return rc;
    // key-frame tables: uploaded from host arrays, or used where they lie when the caller keeps them on the device (the
    // landmark table is copied either way: the evaluation kernels read it long after this call)
    const double *d_kf_t = kf_time, *d_kf_circ = kf_circles;
    if (!on_device) {
        if ((rc = ecb_h2d(ctx, st->kf_t.p, kf_time, (size_t) n_keyframes * 8))) return rc;
        if ((rc = ecb_h2d(ctx, st->kf_circ.p, kf_circles, (size_t) n_keyframes * n_circles * 24))) return rc;
        if ((rc = ecb_h2d(ctx, st->lm_tab.p, landmarks_xyz, (size_t) n_circles * 24))) return rc;
        d_kf_t = (const double *) st->kf_t.p;
        d_kf_circ = (const double *) st->kf_circ.p;
    } else {
        ECB_CUDA(ctx, cudaMemcpyAsync(st->lm_tab.p, landmarks_xyz, (size_t) n_circles * 24, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    AssocArgs a;
    assoc_args(ctx, st, a);
    a.kf_t = d_kf_t;
    a.kf_circ = d_kf_circ;
    a.kf_c32 = (const float2 *) st->kf_c32.p;
    a.K = n_keyframes;
    a.n_circ = n_circles;
    a.n_circ32 = n_circ32;
    a.gate2 = 5 * motion_time_step * 5 * motion_time_step;  // EventCalibSpline.cpp:168
    ECB_PROF_BEGIN(ctx, ECB_STAGE_ASSOC);
    k_circ32<<<(n_keyframes * n_circ32 + 255) / 256, 256, 0, ctx->stream>>>(d_kf_circ, n_keyframes, n_circles,
                                                                           n_circ32, (float2 *) st->kf_c32.p);
    ECB_LAUNCHED(ctx);
    k_assoc_count<<<nb, AS_THREADS, 0, ctx->stream>>>(a, (uint16_t *) st->ev_tag.p, (uint32_t *) st->ev_cnt.p);
    ECB_LAUNCHED(ctx);
    int64_t *d_total = (int64_t *) st->ev_flag.p + nb;
    k_scan_blocks<<<1, 1024, 0, ctx->stream>>>((uint32_t *) st->ev_cnt.p, nb, (int64_t *) st->ev_flag.p, d_total);
    ECB_LAUNCHED(ctx);
    int64_t total = 0;
    if ((rc = ecb_d2h(ctx, &total, d_total, 8))) return rc;
    // time-sorted events + spline ranges in ascending, disjoint order => records come out ordered by (spline, time): the
    // basis pass (k_prepare) is folded into the record write; otherwise k_prepare runs and checks the order
    bool fused = true;
    {
        // The reference adds one residual block per spline whose [front, back] holds the event (EventCalibSpline.cpp:157-192);
        // assoc_one emits at most one.  The two agree while the ranges are disjoint — the reference's own segmentation always
        // is (segments split at gaps > 50 steps, extended by 3 steps) — so overlapping ranges are refused instead of silently
        // dropping the second residual.
        std::vector<std::pair<double, double>> rg;
        size_t ko2 = 0;
        for (int q = 0; q < st->n_splines; ++q) {
            rg.emplace_back(st->knots[ko2], st->knots[ko2 + (size_t) st->n_cp[(size_t) q] + 3]);
            ko2 += (size_t) st->n_cp[(size_t) q] + 4;
        }
        std::sort(rg.begin(), rg.end());
        for (size_t q = 1; q < rg.size(); ++q)
            if (!(rg[q].first > rg[q - 1].second))
                return ecb_fail(ctx, ECB_ERR_UNSUPPORTED,
                                "spline knot ranges overlap ([%g, %g] and [%g, %g]): an event inside both would need one residual "
                                "per spline", rg[q - 1].first, rg[q - 1].second, rg[q].first, rg[q].second);
        size_t ko = 0;
        double prev_end = -1e300;
        for (int q = 0; q < st->n_splines; ++q) {
            const double b = st->knots[ko], e = st->knots[ko + (size_t) st->n_cp[(size_t) q] + 3];
            if (!(b > prev_end)) fused = false;
            prev_end = e;
            ko += (size_t) st->n_cp[(size_t) q] + 4;
        }
    }
    if ((rc = write_assoc_records(ctx, st, a, nb, total, fused))) return rc;
    ECB_PROF_END(ctx, ECB_STAGE_ASSOC);
    if ((rc = ecb_check(ctx, cudaGetLastError(), "association kernels"))) return rc;
    st->n_res = total;
    st->use_circ = fused;
    st->assoc = true;
    st->assoc_K = n_keyframes;
    st->assoc_n_circ = n_circles;
    st->assoc_events_gen = ctx->events_gen;
    st->assoc_kf_t = d_kf_t;
    st->assoc_gate2 = a.gate2;
    if (n_residuals) *n_residuals = total;
    return prepare_records(ctx, st, fused);
}

int ecb_cost_get_association(ecb_ctx *ctx, int64_t *event_index, int32_t *circle_id, int64_t cap) {
    if (!ctx || !ctx->cost) return ECB_ERR_STATE;
    CostState *st = (CostState *) ctx->cost;
    cudaSetDevice(ctx->device);
    const int64_t n = std::min<int64_t>(cap, st->n_res);
    if (n > 0 && event_index)
        ECB_CUDA(ctx, cudaMemcpyAsync(event_index, st->sel_event.p, (size_t) n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (n > 0 && circle_id)
        ECB_CUDA(ctx, cudaMemcpyAsync(circle_id, st->sel_circle.p, (size_t) n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    return ecb_check(ctx, ecb_stream_sync(ctx), "association copy");
}

// ---- launches shared by the host-parameter entry points and the device-side LM loop (ecb_lmdev.cu) ----
}  // extern "C"

static long long exchange_timeout_clocks(ecb_ctx *ctx) {
    static const double secs = getenv("ECB_EXCHANGE_TIMEOUT_S") ? atof(getenv("ECB_EXCHANGE_TIMEOUT_S")) : 30.0;
    // cudaDevAttrClockRate is a live driver query (~1 ms, much more while nvidia-smi polls the device): asked once per device,
    // not per exchange — it was 60 % of a multi-GPU LM iteration (profiles/r2s_lm_exchange_timing.md)
    static int khz_of[64] = {0};
    const int d = ctx->device & 63;
    if (khz_of[d] == 0) {
        int khz = 1965000;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
        khz_of[d] = khz > 0 ? khz : 1965000;
    }
    return (long long) (secs * 1e3 * (double) khz_of[d]);
}

static void fill_ne_args(CostState *st, NeArgs &a, const double *d_params, const int *d_go) {
    a.obs = (const double *) st->obs.p;
    a.lm = (const double *) st->lm.p;
    a.circ = st->use_circ ? (const int *) st->sel_circle.p : nullptr;
    a.lm_tab = (const double *) st->lm_tab.p;
    a.basis = (const double *) st->basis.p;
    a.cp0 = (const int *) st->cp0.p;
    a.items = (const Item *) st->items.p;
    a.n_items = st->n_items;
    a.params = d_params;
    a.total_cp = st->total_cp;
    a.radius = st->radius;
    a.huber = st->huber;
    a.part = (double *) st->part.p;
    a.go = d_go;
}

// k_normal_eq over the residual set with the parameters at d_params (device: intr 9 | rot 4C | trans 3C)
static int launch_normal_eq_kernel(ecb_ctx *ctx, CostState *st, const double *d_params, const int *d_go) {
    NeArgs a;
    fill_ne_args(st, a, d_params, d_go);
    const size_t smem = (size_t) NE_WARPS * TILE_ROWS * TILE_LD * 8;
    // 2 CTAs x 8 warps per SM at 128 registers.  More resident warps for the latency-bound residual / Jacobian phase were tried
    // with 4-warp CTAs: 5 per SM at 96 registers (more spills) 2.10 ms, 4 per SM at 128 registers 1.87 ms, against 1.81 ms
    // (profiles/r2s_ab_normal_eq.jsonl).
    static const int variant = getenv("ECB_NE_VARIANT") ? atoi(getenv("ECB_NE_VARIANT")) : 2;
    void (*kern)(const NeArgs) = st->so3 ? k_normal_eq<1, true> : (variant == 1 ? k_normal_eq<1, false> : k_normal_eq<2, false>);
    ECB_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
    const int grid = std::min((st->n_items + NE_WARPS - 1) / NE_WARPS, ctx->sm_count * ((variant == 1 || st->so3) ? 1 : 2));
    kern<<<grid, NE_THREADS, smem, ctx->stream>>>(a);
    ECB_LAUNCHED(ctx);
    return ECB_OK;
}

static const int *item_start_of(CostState *st) {
    return (const int *) ((const char *) st->items.p + (size_t) std::max(st->n_items, 1) * sizeof(Item));
}

// the span range this rank's residuals contribute to
static void span_range(CostState *st, int &lo, int &hi) {
    lo = 0;
    hi = -1;
    for (int s = 0; s < st->total_spans; ++s)
        if (st->h_span_start[(size_t) s + 1] > st->h_span_start[(size_t) s]) {
            if (hi < 0) lo = s;
            hi = s;
        }
}

// cost-only evaluation at d_params -> *d_cost (device scalar); async
int ecb_cost_dev_eval(ecb_ctx *ctx, const double *d_params, const int *d_go, double *d_cost) {
    CostState *st = (CostState *) ctx->cost;
    int rc;
    if ((rc = ecb_reserve(ctx, st->cost_part, 4096 * 8))) return rc;
    if (st->n_res == 0) {
        ECB_CUDA(ctx, cudaMemsetAsync(d_cost, 0, 8, ctx->stream));
        return ECB_OK;
    }
    const int grid = (int) std::min<int64_t>((st->n_res + 255) / 256, (int64_t) ctx->sm_count * 8);
    ECB_PROF_BEGIN(ctx, ECB_STAGE_COST);
    static const int cost_minb = getenv("ECB_COST_MINB") ? atoi(getenv("ECB_COST_MINB")) : 4;  // 64 registers, 32 warps / SM: 0.35 -> 0.33 ms
    (st->so3 ? k_cost<true, 2> : (cost_minb >= 4 ? k_cost<false, 4> : k_cost<false, 3>))<<<grid, 256, 0, ctx->stream>>>(
        (const double *) st->obs.p, (const double *) st->lm.p, st->use_circ ? (const int *) st->sel_circle.p : nullptr,
        (const double *) st->lm_tab.p, (const double *) st->basis.p, (const int *) st->cp0.p, st->n_res, d_params, st->total_cp,
        st->radius, st->huber, (double *) st->cost_part.p, d_go);
    ECB_LAUNCHED(ctx);
    k_reduce_cost<<<1, 256, 0, ctx->stream>>>((const double *) st->cost_part.p, grid, 1, 0, d_cost, d_go);
    ECB_LAUNCHED(ctx);
    ECB_PROF_END(ctx, ECB_STAGE_COST);
    return ecb_check(ctx, cudaGetLastError(), "cost kernels");
}

// normal equations at d_params -> d_out (packed, this rank's residuals only); async
int ecb_cost_dev_normal_eq(ecb_ctx *ctx, const double *d_params, const int *d_go, double *d_out) {
    CostState *st = (CostState *) ctx->cost;
    if (st->n_items <= 0) return ECB_OK;
    int rc;
    ECB_PROF_BEGIN(ctx, ECB_STAGE_NORMAL_EQ);
    if ((rc = launch_normal_eq_kernel(ctx, st, d_params, d_go))) return rc;
    k_reduce_spans<<<st->total_spans, 192, 0, ctx->stream>>>((const double *) st->part.p, item_start_of(st), st->total_spans, d_out, d_go);
    ECB_LAUNCHED(ctx);
    k_reduce_cost<<<1, 256, 0, ctx->stream>>>((const double *) st->part.p, st->n_items, PART_STRIDE, PART_SC + 3,
                                              d_out + (size_t) st->total_spans * OUT_STRIDE, d_go);
    ECB_LAUNCHED(ctx);
    ECB_PROF_END(ctx, ECB_STAGE_NORMAL_EQ);
    return ecb_check(ctx, cudaGetLastError(), "normal equation kernels");
}

// the same with the inter-GPU sum fused in (all ranks' residuals -> d_out on every rank); the epoch is a device counter
// (d_epoch, already advanced for this exchange) or a host value.  phases as in ecb_cost_normal_eq_exchange.  d_err: sticky
// timeout bits (device word).
int ecb_cost_dev_normal_eq_exchange(ecb_ctx *ctx, const double *d_params, const int *d_go, int rank, int n_ranks,
                                    void *const *recv_buffers, const unsigned long long *d_epoch, unsigned long long epoch,
                                    int phases, double *d_out, unsigned *d_err) {
    CostState *st = (CostState *) ctx->cost;
    int rc;
    if ((rc = ecb_reserve(ctx, st->cost_part, 4096 * 8))) return rc;
    XPeers peers;
    memset(&peers, 0, sizeof peers);
    peers.n_ranks = n_ranks;
    peers.rank = rank;
    for (int p = 0; p < n_ranks; ++p) {
        if (!recv_buffers[p]) return ECB_ERR_ARG;
        peers.base[p] = (double *) recv_buffers[p];
    }
    XCtl x;
    x.go = d_go;
    x.d_epoch = d_epoch;
    x.epoch = epoch;
    x.slot = xslot_doubles(st->total_spans);
    x.n_ranks = n_ranks;
    x.rank = rank;
    int lo, hi;
    span_range(st, lo, hi);
    double *d_cost = (double *) st->cost_part.p + 4001;
    if (phases & ECB_EXCHANGE_SEND) {
        ECB_CUDA(ctx, cudaMemsetAsync(d_cost, 0, 8, ctx->stream));  // (harmless when the launch is gated off)
        if (st->n_items > 0 && hi >= lo) {
            ECB_PROF_BEGIN(ctx, ECB_STAGE_NORMAL_EQ);
            if ((rc = launch_normal_eq_kernel(ctx, st, d_params, d_go))) return rc;
            k_reduce_spans_push<<<hi - lo + 1, 192, 0, ctx->stream>>>((const double *) st->part.p, item_start_of(st), lo, hi, peers, x);
            ECB_LAUNCHED(ctx);
            k_reduce_cost<<<1, 256, 0, ctx->stream>>>((const double *) st->part.p, st->n_items, PART_STRIDE, PART_SC + 3, d_cost, d_go);
            ECB_LAUNCHED(ctx);
            ECB_PROF_END(ctx, ECB_STAGE_NORMAL_EQ);
        }
        k_exchange_signal<<<1, 32, 0, ctx->stream>>>(peers, x, lo, hi, d_cost);
        ECB_LAUNCHED(ctx);
    }
    if (phases & ECB_EXCHANGE_RECV) {
        k_exchange_wait<<<1, 32, 0, ctx->stream>>>(peers.base[rank], x, exchange_timeout_clocks(ctx), d_err);
        ECB_LAUNCHED(ctx);
        k_exchange_sum<<<st->total_spans + 1, 192, 0, ctx->stream>>>(peers.base[rank], x, st->total_spans, d_out, d_err);
        ECB_LAUNCHED(ctx);
    }
    return ecb_check(ctx, cudaGetLastError(), "exchange kernels");
}

// scalar sum over the ranks (device-side LM loop); *d_value: this rank's part in, the sum out
int ecb_cost_dev_scalar_exchange(ecb_ctx *ctx, const int *d_go, int rank, int n_ranks, void *const *recv_buffers,
                                 const unsigned long long *d_epoch, double *d_value, unsigned *d_err) {
    CostState *st = (CostState *) ctx->cost;
    XPeers peers;
    memset(&peers, 0, sizeof peers);
    peers.n_ranks = n_ranks;
    peers.rank = rank;
    for (int p = 0; p < n_ranks; ++p) peers.base[p] = (double *) recv_buffers[p];
    XCtl x;
    x.go = d_go;
    x.d_epoch = d_epoch;
    x.epoch = 0;
    x.slot = xslot_doubles(st->total_spans);
    x.n_ranks = n_ranks;
    x.rank = rank;
    k_exchange_scalar<<<1, 32, 0, ctx->stream>>>(peers, x, 2 * (size_t) n_ranks * x.slot, d_value, exchange_timeout_clocks(ctx), d_err);
    ECB_LAUNCHED(ctx);
    return ecb_check(ctx, cudaGetLastError(), "scalar exchange");
}

double *ecb_cost_params_buffer(ecb_ctx *ctx, size_t *doubles) {  // the context's parameter upload buffer (intr | rot | trans)
    CostState *st = (CostState *) ctx->cost;
    const size_t n = 9 + 7 * (size_t) st->total_cp;
    if (ecb_reserve(ctx, st->params, n * 8)) return nullptr;
    if (doubles) *doubles = n;
    return (double *) st->params.p;
}

extern "C" {

int ecb_cost_eval(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, double *cost) {
    if (!ctx || !ctx->cost || !intrinsics || !rot_cp || !trans_cp || !cost) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    CostState *st = (CostState *) ctx->cost;
    int rc;
    if ((rc = upload_params(ctx, st, intrinsics, rot_cp, trans_cp))) return rc;
    if ((rc = ecb_reserve(ctx, st->cost_part, 4096 * 8))) return rc;
    *cost = 0.0;
    if (st->n_res == 0) return ECB_OK;
    if ((rc = ecb_cost_dev_eval(ctx, (const double *) st->params.p, nullptr, (double *) st->cost_part.p + 4000))) return rc;
    return ecb_d2h(ctx, cost, (double *) st->cost_part.p + 4000, 8);
}

// Packed result (device or host): per span s  [H 33x33 full symmetric | g 33], then [cost, 0].
// d_out (device pointer, may be NULL -> internal buffer); h_out (host, may be NULL).
int ecb_cost_normal_eq(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, void *d_out,
                       double *h_out, double *cost) {
    if (!ctx || !ctx->cost || !intrinsics || !rot_cp || !trans_cp) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    CostState *st = (CostState *) ctx->cost;
    int rc;
    if ((rc = upload_params(ctx, st, intrinsics, rot_cp, trans_cp))) return rc;
    const size_t n_out = (size_t) st->total_spans * OUT_STRIDE + 2;
    if ((rc = ecb_reserve(ctx, st->out, (n_out + 8) * 8))) return rc;
    double *out = d_out ? (double *) d_out : (double *) st->out.p;
    ECB_CUDA(ctx, cudaMemsetAsync(out, 0, n_out * 8, ctx->stream));
    if ((rc = ecb_cost_dev_normal_eq(ctx, (const double *) st->params.p, nullptr, out))) return rc;
    if (h_out) {
        if ((rc = ecb_d2h(ctx, h_out, out, n_out * 8))) return rc;
        if (cost) *cost = h_out[(size_t) st->total_spans * OUT_STRIDE];
    } else if (cost) {
        return ecb_d2h(ctx, cost, out + (size_t) st->total_spans * OUT_STRIDE, 8);
    }
    return ECB_OK;
}

}  // extern "C"

// ---- residual and reprojection reports ----
// the metric m of every record at the point already uploaded to st->params -> out (device, n_res doubles); d_invalid (optional,
// zeroed here) counts the NaN values; async
template <class Metric>
static int launch_record_report(ecb_ctx *ctx, CostState *st, const Metric &m, double *out, unsigned long long *d_invalid) {
    if (d_invalid) ECB_CUDA(ctx, cudaMemsetAsync(d_invalid, 0, 8, ctx->stream));
    if (st->n_res == 0) return ECB_OK;
    const int grid = (int) std::min<int64_t>((st->n_res + 255) / 256, (int64_t) ctx->sm_count * 8);
    (st->so3 ? k_record_report<1, Metric> : k_record_report<0, Metric>)<<<grid, 256, 0, ctx->stream>>>(
        (const double *) st->obs.p, (const double *) st->lm.p, st->use_circ ? (const int *) st->sel_circle.p : nullptr,
        (const double *) st->lm_tab.p, (const double *) st->basis.p, (const int *) st->cp0.p, st->n_res,
        (const double *) st->params.p, st->total_cp, m, out, d_invalid);
    ECB_LAUNCHED(ctx);
    return ecb_check(ctx, cudaGetLastError(), "k_record_report");
}

// ecb_cost_residuals and ecb_cost_reprojection_errors
template <class Metric>
static int record_report(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, double *d_out,
                         double *h_out, int64_t *n_invalid) {
    if (!ctx || !intrinsics || !rot_cp || !trans_cp) return ECB_ERR_ARG;
    if (!ctx->cost) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_cost_setup first");
    cudaSetDevice(ctx->device);
    CostState *st = (CostState *) ctx->cost;
    if (st->n_res > 0xFFFFFFFFll) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "%s report over 2^32 or more records", Metric::report);
    int rc;
    if ((rc = upload_params(ctx, st, intrinsics, rot_cp, trans_cp))) return rc;
    double *out = d_out;
    if (!out) {
        if ((rc = ecb_reserve(ctx, st->rep_r, (size_t) std::max<int64_t>(st->n_res, 1) * 8))) return rc;
        out = (double *) st->rep_r.p;
    }
    unsigned long long *d_invalid = nullptr;
    if (n_invalid) {
        if ((rc = ecb_reserve(ctx, st->rep_io, 8))) return rc;
        d_invalid = (unsigned long long *) st->rep_io.p;
    }
    if ((rc = launch_record_report(ctx, st, Metric::at(st, intrinsics), out, d_invalid))) return rc;
    if (h_out && (rc = ecb_d2h(ctx, h_out, out, (size_t) st->n_res * 8))) return rc;
    if (n_invalid) {
        unsigned long long c = 0;
        if ((rc = ecb_d2h(ctx, &c, d_invalid, 8))) return rc;
        *n_invalid = (int64_t) c;
    }
    return ECB_OK;
}

// The records come from an association (else ECB_ERR_STATE with the message `none`); with `events`, of the events loaded now;
// with n_keyframes, over that many key frames (else ECB_ERR_ARG).
static int check_association(ecb_ctx *ctx, const CostState *st, const char *none, bool events, const int *n_keyframes) {
    if (!st->assoc) return ecb_fail(ctx, ECB_ERR_STATE, "%s", none);
    if (events && st->assoc_events_gen != ctx->events_gen) return ecb_fail(ctx, ECB_ERR_STATE, "events were loaded after the association");
    if (n_keyframes && *n_keyframes != st->assoc_K)
        return ecb_fail(ctx, ECB_ERR_ARG, "%d key frames given, the association used %d", *n_keyframes, st->assoc_K);
    return ECB_OK;
}

// The grouping shared by the residual and the reprojection report (ecb_cost_residual_groups): group_layout checks the
// arguments, counts the groups (*G; *n_groups is always set) and fills the key arguments; *query is set for a pure size query.
static int group_layout(ecb_ctx *ctx, CostState *st, int by, const double *kf_time, int n_keyframes, int cell_px, bool have_groups,
                        int cap, int *n_groups, GroupKeyArgs &a, int64_t *G, bool *query) {
    if (by != ECB_RESIDUALS_BY_KEYFRAME && by != ECB_RESIDUALS_BY_CIRCLE && by != ECB_RESIDUALS_BY_SENSOR_CELL)
        return ecb_fail(ctx, ECB_ERR_ARG, "unknown residual grouping %d", by);
    if (cell_px < 1) return ecb_fail(ctx, ECB_ERR_ARG, "cell size %d px < 1", cell_px);
    if (by == ECB_RESIDUALS_BY_KEYFRAME && !kf_time) return ecb_fail(ctx, ECB_ERR_ARG, "grouping by key frame needs the stamps");
    if (!st) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_cost_setup first");
    memset(&a, 0, sizeof a);
    a.by = by;
    if (by == ECB_RESIDUALS_BY_KEYFRAME || by == ECB_RESIDUALS_BY_CIRCLE) {
        const bool kf = by == ECB_RESIDUALS_BY_KEYFRAME;
        int rc;
        if ((rc = check_association(ctx, st, "residuals of ecb_cost_set_residuals have no key frame or circle: associate first", kf,
                                    kf ? &n_keyframes : nullptr)))
            return rc;
        *G = kf ? st->assoc_K : st->assoc_n_circ;
    } else {
        if (ctx->width <= 0 || ctx->height <= 0) return ecb_fail(ctx, ECB_ERR_STATE, "grouping by sensor cell needs ecb_set_sensor");
        a.width = ctx->width;
        a.height = ctx->height;
        a.cell = cell_px;
        a.ncx = (ctx->width + cell_px - 1) / cell_px;
        *G = (int64_t) a.ncx * ((ctx->height + cell_px - 1) / cell_px);
    }
    if (n_groups) *n_groups = (int) *G;
    *query = !have_groups && cap == 0;
    if (*query) return ECB_OK;
    if (cap < *G || !have_groups) return ecb_fail(ctx, ECB_ERR_ARG, "%lld groups do not fit cap %d", (long long) *G, cap);
    if (st->n_res > 0xFFFFFFFFll) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "residual report over 2^32 or more records");
    return ECB_OK;
}

// group_sort: the (group, record index) keys of the n_res >= 1 records, sorted with the stable radix sort, and the group bounds
// st->rep_start[0 .. G + 1]; *sidx: the record indices in group order (record order inside a group).  Async.
static int group_sort(ecb_ctx *ctx, CostState *st, GroupKeyArgs a, int64_t G, const double *kf_time, const uint32_t **sidx) {
    int rc;
    const int64_t n = st->n_res;
    const size_t un = (size_t) n;
    for (int q = 0; q < 2; ++q) {
        if ((rc = ecb_reserve(ctx, st->rep_key[q], un * 8))) return rc;
        if ((rc = ecb_reserve(ctx, st->rep_idx[q], un * 4))) return rc;
    }
    if ((rc = ecb_reserve(ctx, st->rep_hist, gh_radix_hist_bytes(n)))) return rc;
    if ((rc = ecb_reserve(ctx, st->rep_start, ((size_t) G + 2) * 8))) return rc;
    if (a.by == ECB_RESIDUALS_BY_KEYFRAME) {
        if ((rc = ecb_reserve(ctx, st->rep_kf, (size_t) G * 8))) return rc;
        if ((rc = ecb_h2d(ctx, st->rep_kf.p, kf_time, (size_t) G * 8))) return rc;
    }
    a.sel_event = (const int64_t *) st->sel_event.p;
    a.sel_circle = (const int *) st->sel_circle.p;
    a.ev_t = (const double *) ctx->ev_t.p;
    a.kf_t = (const double *) st->rep_kf.p;
    a.K = (int) G;
    a.obs = (const double *) st->obs.p;
    a.outside = (uint32_t) G;
    uint64_t *key[2] = {(uint64_t *) st->rep_key[0].p, (uint64_t *) st->rep_key[1].p};
    uint32_t *idx[2] = {(uint32_t *) st->rep_idx[0].p, (uint32_t *) st->rep_idx[1].p};
    const int grid = (int) std::min<int64_t>((n + 255) / 256, (int64_t) ctx->sm_count * 8);
    k_group_keys<<<grid, 256, 0, ctx->stream>>>(a, n, key[0], idx[0]);
    ECB_LAUNCHED(ctx);
    int bits = 8;
    while (bits < 64 && ((uint64_t) G >> bits)) bits += 8;  // keys 0 .. G
    int res = 0;
    if ((rc = gh_radix_sort(ctx, key, idx, n, bits, (uint32_t *) st->rep_hist.p, &res))) return rc;
    k_group_start<<<(unsigned) ((G + 2 + 127) / 128), 128, 0, ctx->stream>>>(key[res], n, (int) G + 1, (int64_t *) st->rep_start.p);
    ECB_LAUNCHED(ctx);
    *sidx = idx[res];
    return ecb_check(ctx, cudaGetLastError(), "group kernels");
}

// ecb_cost_residual_groups and ecb_cost_reprojection_groups
template <class Metric, class Stats = typename Metric::Stats, class Group = typename Stats::Group>
static int group_report(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, int by,
                        const double *kf_time, int n_keyframes, int cell_px, Group *groups, int cap, int *n_groups, Group *total) {
    if (!ctx || !intrinsics || !rot_cp || !trans_cp) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    CostState *st = (CostState *) ctx->cost;
    GroupKeyArgs a;
    int64_t G = 0;
    bool query = false;
    int rc;
    if ((rc = group_layout(ctx, st, by, kf_time, n_keyframes, cell_px, groups != nullptr, cap, n_groups, a, &G, &query))) return rc;
    if (query) return ECB_OK;
    const int64_t n = st->n_res;
    const Metric m = Metric::at(st, intrinsics);
    std::vector<Group> h((size_t) G + 1);
    memset(h.data(), 0, h.size() * sizeof(Group));
    if (n > 0) {
        if ((rc = upload_params(ctx, st, intrinsics, rot_cp, trans_cp))) return rc;
        if ((rc = ecb_reserve(ctx, st->rep_r, (size_t) n * 8))) return rc;
        if ((rc = ecb_reserve(ctx, st->rep_out, ((size_t) G + 1) * sizeof(Group)))) return rc;
        if ((rc = launch_record_report(ctx, st, m, (double *) st->rep_r.p, nullptr))) return rc;
        const uint32_t *sidx = nullptr;
        if ((rc = group_sort(ctx, st, a, G, kf_time, &sidx))) return rc;
        k_group_stats<Stats><<<(unsigned) (G + 1), RG_THREADS, 0, ctx->stream>>>((const double *) st->rep_r.p, sidx,
                                                                               (const int64_t *) st->rep_start.p, m.stats(),
                                                                               (Group *) st->rep_out.p);
        ECB_LAUNCHED(ctx);
        if ((rc = ecb_check(ctx, cudaGetLastError(), "k_group_stats"))) return rc;
        if ((rc = ecb_d2h(ctx, h.data(), st->rep_out.p, h.size() * sizeof(Group)))) return rc;
    }
    memcpy(groups, h.data(), (size_t) G * sizeof(Group));
    if (total) {  // groups 0 .. G-1 and the records outside every group, in group order
        Stats s = m.stats();
        for (const Group &q : h) s.merge(Stats{q});
        *total = s.result();
    }
    return ECB_OK;
}

extern "C" {

int ecb_cost_residuals(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, double *d_out,
                       double *h_out) {
    return record_report<ResidualMetric>(ctx, intrinsics, rot_cp, trans_cp, d_out, h_out, nullptr);
}

int ecb_cost_reprojection_errors(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp,
                                 double *d_out, double *h_out, int64_t *n_invalid) {
    return record_report<RimReprojectionMetric>(ctx, intrinsics, rot_cp, trans_cp, d_out, h_out, n_invalid);
}

int ecb_cost_residual_groups(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, int by,
                             const double *kf_time, int n_keyframes, int cell_px, ecb_residual_group *groups, int cap,
                             int *n_groups, ecb_residual_group *total) {
    return group_report<ResidualMetric>(ctx, intrinsics, rot_cp, trans_cp, by, kf_time, n_keyframes, cell_px, groups, cap,
                                         n_groups, total);
}

int ecb_cost_reprojection_groups(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, int by,
                                 const double *kf_time, int n_keyframes, int cell_px, ecb_reprojection_group *groups, int cap,
                                 int *n_groups, ecb_reprojection_group *total) {
    return group_report<RimReprojectionMetric>(ctx, intrinsics, rot_cp, trans_cp, by, kf_time, n_keyframes, cell_px, groups, cap,
                                               n_groups, total);
}

// ---- outlier rejection ----
int ecb_cost_reject(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, double max_abs_residual,
                    const double *kf_time, const uint8_t *drop_keyframe, int n_keyframes, int64_t *n_kept, int64_t *n_removed) {
    if (!ctx || !intrinsics || !rot_cp || !trans_cp) return ECB_ERR_ARG;
    if (!(max_abs_residual >= 0.0)) return ecb_fail(ctx, ECB_ERR_ARG, "max_abs_residual %g is NaN or negative", max_abs_residual);
    if (drop_keyframe && !kf_time) return ecb_fail(ctx, ECB_ERR_ARG, "a key-frame mask needs the key-frame stamps");
    if (!ctx->cost) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_cost_setup first");
    cudaSetDevice(ctx->device);
    CostState *st = (CostState *) ctx->cost;
    int rc;
    if (drop_keyframe &&
        (rc = check_association(ctx, st, "residuals of ecb_cost_set_residuals have no key frame: associate first", true, &n_keyframes)))
        return rc;
    const int64_t n = st->n_res;
    if (n > 0xFFFFFFFFll) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "outlier rejection over 2^32 or more records");
    if (n_kept) *n_kept = n;
    if (n_removed) *n_removed = 0;
    if (n == 0) return ECB_OK;
    const int nb = (int) ((n + AS_THREADS - 1) / AS_THREADS);
    // r_k as ecb_cost_residuals returns it; the association's scratch holds the keep flags, block counts and offsets
    if ((rc = upload_params(ctx, st, intrinsics, rot_cp, trans_cp))) return rc;
    if ((rc = ecb_reserve(ctx, st->rep_r, (size_t) n * 8))) return rc;
    if ((rc = ecb_reserve(ctx, st->ev_tag, (size_t) n + 16))) return rc;
    if ((rc = ecb_reserve(ctx, st->ev_cnt, (size_t) nb * 4 + 16))) return rc;
    if ((rc = ecb_reserve(ctx, st->ev_flag, (size_t) nb * 8 + 16))) return rc;
    if ((rc = launch_record_report(ctx, st, ResidualMetric::at(st, intrinsics), (double *) st->rep_r.p, nullptr))) return rc;
    RejectArgs a;
    memset(&a, 0, sizeof a);
    a.r = (const double *) st->rep_r.p;
    a.max_abs = max_abs_residual;
    a.n = n;
    if (drop_keyframe) {  // the mask and the stamps share one upload
        const size_t K = (size_t) n_keyframes;
        std::vector<uint8_t> up(K * 8 + K);
        memcpy(up.data(), kf_time, K * 8);
        memcpy(up.data() + K * 8, drop_keyframe, K);
        if ((rc = ecb_reserve(ctx, st->rep_kf, up.size()))) return rc;
        if ((rc = ecb_h2d(ctx, st->rep_kf.p, up.data(), up.size()))) return rc;
        a.kf_t = (const double *) st->rep_kf.p;
        a.drop = (const uint8_t *) st->rep_kf.p + K * 8;
        a.K = n_keyframes;
        a.sel_event = (const int64_t *) st->sel_event.p;
        a.ev_t = (const double *) ctx->ev_t.p;
    }
    uint8_t *keep = (uint8_t *) st->ev_tag.p;
    int64_t *off = (int64_t *) st->ev_flag.p, *d_total = off + nb;
    k_reject_count<<<nb, AS_THREADS, 0, ctx->stream>>>(a, keep, (uint32_t *) st->ev_cnt.p);
    ECB_LAUNCHED(ctx);
    k_scan_blocks<<<1, 1024, 0, ctx->stream>>>((uint32_t *) st->ev_cnt.p, nb, off, d_total);
    ECB_LAUNCHED(ctx);
    int64_t kept = 0;
    if ((rc = ecb_d2h(ctx, &kept, d_total, 8))) return rc;
    if (n_kept) *n_kept = kept;
    if (n_removed) *n_removed = n - kept;
    if (kept == n) return ECB_OK;  // nothing removed: the records stay as they are, byte for byte
    // every array the path holds: obs / basis / cp0 / span always, event and circle of an association, landmark / time /
    // spline of explicit or unfused records
    DevBuf *live[9] = {&st->obs, &st->basis, &st->cp0, &st->span, &st->sel_event, &st->sel_circle, &st->lm, &st->tt, &st->spl};
    const size_t esz[9] = {16, 32, 4, 4, 8, 4, 24, 8, 4};
    bool moved[9];
    for (int i = 0; i < 9; ++i) moved[i] = i < 4 || (i < 6 ? st->assoc : !st->use_circ);
    const size_t nk = (size_t) std::max<int64_t>(kept, 1);
    void *src[9] = {}, *dst[9] = {};
    for (int i = 0; i < 9; ++i) {
        if (!moved[i]) continue;
        if ((rc = ecb_reserve(ctx, st->rej[i], nk * esz[i]))) return rc;
        src[i] = live[i]->p;
        dst[i] = st->rej[i].p;
    }
    auto ptrs = [](void *const *p) {
        RecordPtrs r;
        r.obs = (double2 *) p[0];
        r.basis = (double4 *) p[1];
        r.cp0 = (int *) p[2];
        r.span = (int *) p[3];
        r.sel_event = (int64_t *) p[4];
        r.sel_circle = (int *) p[5];
        r.lm = (double *) p[6];
        r.tt = (double *) p[7];
        r.spl = (int *) p[8];
        return r;
    };
    k_reject_write<<<nb, AS_THREADS, 0, ctx->stream>>>(keep, off, n, ptrs(src), ptrs(dst));
    ECB_LAUNCHED(ctx);
    if ((rc = ecb_check(ctx, cudaGetLastError(), "outlier rejection kernels"))) return rc;
    for (int i = 0; i < 9; ++i)
        if (moved[i]) std::swap(*live[i], st->rej[i]);
    st->n_res = kept;
    if ((rc = prepare_records(ctx, st, /*have_basis=*/true))) return rc;
    return ecb_check(ctx, ecb_stream_sync(ctx), "outlier rejection");
}

// ---- re-association ----
int ecb_cost_reassociate(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, double gate_px,
                         double max_dt, int64_t *n_residuals, int64_t *n_same, int64_t *n_changed, int64_t *n_new,
                         int64_t *n_lost) {
    if (!ctx || !intrinsics || !rot_cp || !trans_cp) return ECB_ERR_ARG;
    if (!(gate_px > 0.0)) return ecb_fail(ctx, ECB_ERR_ARG, "gate_px %g is NaN or not positive", gate_px);
    if (!(max_dt >= 0.0)) return ecb_fail(ctx, ECB_ERR_ARG, "max_dt %g is NaN or negative", max_dt);
    if (!ctx->cost) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_cost_setup first");
    cudaSetDevice(ctx->device);
    CostState *st = (CostState *) ctx->cost;
    int rc;
    if ((rc = check_association(ctx, st, "the records do not come from an association: associate first", true, nullptr))) return rc;
    if (st->n_res > 0xFFFFFFFFll) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "re-association of 2^32 or more records");
    const int64_t n = ctx->n_events, n_prev = st->n_res;  // n < 2^32: the association checked it for these events
    const int nb = (int) ((n + AS_THREADS - 1) / AS_THREADS);
    if ((rc = upload_params(ctx, st, intrinsics, rot_cp, trans_cp))) return rc;
    if ((rc = ecb_reserve(ctx, st->ev_cnt, (size_t) nb * 4 + 16))) return rc;
    if ((rc = ecb_reserve(ctx, st->ev_tag, (size_t) n * 2 + 16))) return rc;
    if ((rc = ecb_reserve(ctx, st->ev_flag, (size_t) nb * 8 + 48))) return rc;
    // block offsets | total | same, changed, new: one read-back
    int64_t *off = (int64_t *) st->ev_flag.p, *d_total = off + nb;
    ECB_CUDA(ctx, cudaMemsetAsync(d_total + 1, 0, 24, ctx->stream));
    ReassocArgs r;
    memset(&r, 0, sizeof r);
    assoc_args(ctx, st, r.as);
    r.as.kf_t = st->assoc_kf_t;
    r.as.K = st->assoc_K;
    r.as.n_circ = st->assoc_n_circ;
    r.as.gate2 = st->assoc_gate2;
    r.max_dt = max_dt;
    r.params = (const double *) st->params.p;
    r.total_cp = st->total_cp;
    r.fold = ecb_inverse_radial_fold_host(intrinsics + 4);
    r.radius = st->radius;
    r.gate_px = gate_px;
    r.prev_event = (const int64_t *) st->sel_event.p;
    r.prev_circle = (const int *) st->sel_circle.p;
    r.n_prev = n_prev;
    r.counts = (unsigned long long *) (d_total + 1);
    (st->so3 ? k_reassoc_count<1> : k_reassoc_count<0>)<<<nb, AS_THREADS, 0, ctx->stream>>>(r, (uint16_t *) st->ev_tag.p,
                                                                                           (uint32_t *) st->ev_cnt.p);
    ECB_LAUNCHED(ctx);
    k_scan_blocks<<<1, 1024, 0, ctx->stream>>>((uint32_t *) st->ev_cnt.p, nb, off, d_total);
    ECB_LAUNCHED(ctx);
    int64_t h[4] = {0, 0, 0, 0};  // total, same, changed, new
    if ((rc = ecb_d2h(ctx, h, d_total, sizeof h))) return rc;
    // the previous records have been read: the new ones may take their buffers
    if ((rc = write_assoc_records(ctx, st, r.as, nb, h[0], st->use_circ))) return rc;
    if ((rc = ecb_check(ctx, cudaGetLastError(), "re-association kernels"))) return rc;
    st->n_res = h[0];
    if ((rc = prepare_records(ctx, st, st->use_circ))) return rc;
    if ((rc = ecb_check(ctx, ecb_stream_sync(ctx), "re-association"))) return rc;
    if (n_residuals) *n_residuals = h[0];
    if (n_same) *n_same = h[1];
    if (n_changed) *n_changed = h[2];
    if (n_new) *n_new = h[3];
    if (n_lost) *n_lost = n_prev - h[1] - h[2];
    return ECB_OK;
}

// ---- reprojection report ----
int ecb_inverse_radial_fold(const double *k, double *rho_fold) {
    if (!k || !rho_fold) return ECB_ERR_ARG;
    *rho_fold = ecb_inverse_radial_fold_host(k).rho;
    return ECB_OK;
}

int ecb_keyframe_reprojection(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp,
                              const double *kf_time, const double *kf_circles, int n_keyframes, int n_circles,
                              const double *landmarks_xyz, double *proj, double *err, ecb_reprojection_group *total) {
    if (!ctx || !intrinsics || !rot_cp || !trans_cp || !kf_time || !kf_circles || !landmarks_xyz || n_keyframes < 1 ||
        n_circles < 1)
        return ECB_ERR_ARG;
    if (!ctx->cost) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_cost_setup first");
    cudaSetDevice(ctx->device);
    CostState *st = (CostState *) ctx->cost;
    const size_t K = (size_t) n_keyframes, nc = (size_t) n_circles, m = K * nc;
    int rc;
    if ((rc = upload_params(ctx, st, intrinsics, rot_cp, trans_cp))) return rc;
    // staging: kf_t K | circles 3 m | landmarks 3 nc | proj 2 m | err m
    if ((rc = ecb_reserve(ctx, st->rep_io, (K + 6 * m + 3 * nc) * 8))) return rc;
    double *d_t = (double *) st->rep_io.p, *d_c = d_t + K, *d_l = d_c + 3 * m, *d_p = d_l + 3 * nc, *d_e = d_p + 2 * m;
    if ((rc = ecb_h2d(ctx, d_t, kf_time, K * 8))) return rc;
    if ((rc = ecb_h2d(ctx, d_c, kf_circles, 3 * m * 8))) return rc;
    if ((rc = ecb_h2d(ctx, d_l, landmarks_xyz, 3 * nc * 8))) return rc;
    EcbSplineView sv;
    ecb_cost_spline_view(ctx, &sv);
    const EcbFold fold = ecb_inverse_radial_fold_host(intrinsics + 4);
    (st->so3 ? k_keyframe_reproj<1> : k_keyframe_reproj<0>)<<<(unsigned) ((m + 127) / 128), 128, 0, ctx->stream>>>(
        d_t, d_c, d_l, n_keyframes, n_circles, sv, (const double *) st->params.p, fold, d_p, d_e);
    ECB_LAUNCHED(ctx);
    if ((rc = ecb_check(ctx, cudaGetLastError(), "k_keyframe_reproj"))) return rc;
    std::vector<double> h(3 * m);
    if ((rc = ecb_d2h(ctx, h.data(), d_p, 3 * m * 8))) return rc;
    if (proj) memcpy(proj, h.data(), 2 * m * 8);
    if (err) memcpy(err, h.data() + 2 * m, m * 8);
    if (total) {  // the present features in (key frame, circle) order
        ecb_reprojection_group s;
        memset(&s, 0, sizeof s);
        for (size_t i = 0; i < m; ++i) {
            if (!(kf_circles[3 * i + 2] >= 0.0)) continue;  // absent (as in k_keyframe_reproj)
            const double e = h[2 * m + i];
            if (std::isnan(e)) {
                ++s.n_invalid;
                continue;
            }
            ++s.count;
            s.sum += e;
            s.sum_sq += e * e;
            s.max_abs = std::max(s.max_abs, e);
        }
        *total = s;
    }
    return ECB_OK;
}

// ---- fused reduce + exchange (multi-GPU) ----
size_t ecb_exchange_buffer_bytes(ecb_ctx *ctx, int n_ranks) {
    if (!ctx || !ctx->cost || n_ranks < 1) return 0;
    CostState *st = (CostState *) ctx->cost;
    // two parity blocks of n_ranks span slots, then two parity blocks of n_ranks (epoch, value) scalar slots
    return (2 * (size_t) n_ranks * xslot_doubles(st->total_spans) + 4 * (size_t) n_ranks + 8) * 8;
}

int ecb_cost_normal_eq_exchange(ecb_ctx *ctx, const double *intrinsics, const double *rot_cp, const double *trans_cp, int rank,
                                int n_ranks, void *const *recv_buffers, uint64_t epoch, int phases, void *d_out, double *cost) {
    if (!ctx || !ctx->cost || !intrinsics || !rot_cp || !trans_cp || !recv_buffers || !d_out) return ECB_ERR_ARG;
    if (!(phases & 3)) return ECB_ERR_ARG;
    if (n_ranks < 1 || n_ranks > ECB_MAX_PEERS || rank < 0 || rank >= n_ranks || epoch == 0) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    CostState *st = (CostState *) ctx->cost;
    int rc;
    if ((rc = upload_params(ctx, st, intrinsics, rot_cp, trans_cp))) return rc;
    if ((rc = ecb_reserve(ctx, st->cost_part, 4096 * 8))) return rc;
    // Epochs on the wire never repeat for a receive buffer: a caller that restarts its sequence (a second LM run on the same
    // buffers begins at 1 again) starts a new generation, so a header left over from the previous run cannot satisfy the wait.
    // Every rank sees the same epoch sequence, hence the same generations.  (SEND and RECV of one exchange carry one epoch.)
    if ((phases & ECB_EXCHANGE_SEND) && epoch <= st->xch_last_epoch) ++st->xch_generation;
    if (phases & ECB_EXCHANGE_SEND) st->xch_last_epoch = epoch;
    const unsigned long long wire = ((unsigned long long) st->xch_generation << 40) | (unsigned long long) (epoch & 0xFFFFFFFFFFull);
    // the parity must follow the caller's epoch (double buffering), generations keep it: shift left by one, parity in bit 0
    const unsigned long long wire_epoch = (wire << 1) | (epoch & 1ull);
    unsigned *d_err = (unsigned *) ((double *) st->cost_part.p + 4002);
    if (phases & ECB_EXCHANGE_SEND) ECB_CUDA(ctx, cudaMemsetAsync(d_err, 0, 4, ctx->stream));
    if ((rc = ecb_cost_dev_normal_eq_exchange(ctx, (const double *) st->params.p, nullptr, rank, n_ranks, recv_buffers, nullptr,
                                              wire_epoch, phases, (double *) d_out, d_err)))
        return rc;
    if (!(phases & ECB_EXCHANGE_RECV)) return ECB_OK;
    if (cost) {
        double hc[2];
        if ((rc = ecb_d2h(ctx, hc, (double *) d_out + (size_t) st->total_spans * OUT_STRIDE, 8))) return rc;
        unsigned herr = 0;
        if ((rc = ecb_d2h(ctx, &herr, d_err, 4))) return rc;
        if (herr) return ecb_fail(ctx, ECB_ERR_STATE, "normal-equation exchange timed out waiting for ranks (mask 0x%x)", herr);
        *cost = hc[0];
    }
    // cost == NULL: nothing is read back here; a timeout leaves NaN in the cost slot of d_out (k_exchange_sum), which every
    // consumer of the packed buffer sees
    return ECB_OK;
}

}  // extern "C"
