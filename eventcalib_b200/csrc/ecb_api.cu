// C ABI of libecb: context, ingest, batched front end, DBSCAN::Run boundary, batched circle fit.
// See include/eventcalib_b200.h for the reference interface each entry point replaces.
#include <sched.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "ecb_window.cuh"

int ecb_fail(ecb_ctx *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return code;
}

int ecb_check(ecb_ctx *ctx, cudaError_t e, const char *what) {
    if (e == cudaSuccess) return ECB_OK;
    return ecb_fail(ctx, ECB_ERR_CUDA, "CUDA error %s: %s", what, cudaGetErrorString(e));
}

int ecb_reserve(ecb_ctx *ctx, DevBuf &b, size_t bytes) {
    if (bytes <= b.cap && b.p) return ECB_OK;
    if (b.p) {
        ecb_stream_sync(ctx);
        cudaFree(b.p);
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = bytes + bytes / 8 + 256;
    ECB_CUDA(ctx, cudaMalloc(&b.p, want));
    b.cap = want;
    return ECB_OK;
}

__global__ void k_pull(uint32_t *__restrict__ dst, const uint32_t *__restrict__ src, size_t words, size_t bytes) {
    for (size_t i = (size_t) blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (size_t) gridDim.x * blockDim.x)
        dst[i] = src[i];
    if (blockIdx.x == 0 && threadIdx.x < (bytes & 3))
        ((uint8_t *) dst)[words * 4 + threadIdx.x] = ((const uint8_t *) src)[words * 4 + threadIdx.x];
}

cudaError_t ecb_stream_sync(ecb_ctx *ctx) {
    if (!ctx->sync_mode || !ctx->sync_ev) return cudaStreamSynchronize(ctx->stream);
    cudaError_t e = cudaEventRecord(ctx->sync_ev, ctx->stream);
    if (e != cudaSuccess) return e;
    if (ctx->sync_mode == 1) return cudaEventSynchronize(ctx->sync_ev);  // sleeps until the driver wakes the thread
    while ((e = cudaEventQuery(ctx->sync_ev)) == cudaErrorNotReady) sched_yield();  // polls, but gives the core away in between
    return e;
}

static int reserve_pinned(ecb_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->pinned_cap) return ECB_OK;
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    ctx->pinned = nullptr;
    ctx->pinned_cap = 0;
    bytes += bytes / 4 + 4096;
    ECB_CUDA(ctx, cudaHostAlloc(&ctx->pinned, bytes, cudaHostAllocMapped));
    ctx->pinned_cap = bytes;
    return ECB_OK;
}

// Device -> host copy + stream synchronisation through the context's pinned staging buffer: a cudaMemcpyAsync into
// pageable memory takes the driver's slow staged path and serialises against other threads' transfers.
int ecb_d2h(ecb_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (bytes == 0) return ecb_check(ctx, ecb_stream_sync(ctx), "stream synchronize");
    if (bytes > ((size_t) 256 << 20)) {
        ECB_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        return ecb_check(ctx, ecb_stream_sync(ctx), "device to host copy");
    }
    int rc = reserve_pinned(ctx, bytes);
    if (rc) return rc;
    if (bytes <= ((size_t) 1 << 20) && !((uintptr_t) src & 3u)) {
        // small results never touch the copy engines either: a kernel stores them into the (device-mapped) pinned buffer,
        // so a window table or a scalar cannot queue behind another context's bulk record DMA
        void *dpin = nullptr;
        ECB_CUDA(ctx, cudaHostGetDevicePointer(&dpin, ctx->pinned, 0));
        const size_t words = bytes >> 2;
        const int grid = (int) std::min<size_t>((words + 255) / 256 + 1, 128);
        k_pull<<<grid, 256, 0, ctx->stream>>>((uint32_t *) dpin, (const uint32_t *) src, words, bytes);
        ECB_LAUNCHED(ctx);
        ECB_CUDA(ctx, cudaGetLastError());
    } else {
        ECB_CUDA(ctx, cudaMemcpyAsync(ctx->pinned, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    ECB_CUDA(ctx, ecb_stream_sync(ctx));
    ctx->up_off = 0;  // every staged upload has been pulled
    memcpy(dst, ctx->pinned, bytes);
    return ECB_OK;
}

int ecb_h2d(ecb_ctx *ctx, void *dst, const void *src, size_t bytes) {
    if (bytes == 0) return ECB_OK;
    if (bytes > ((size_t) 8 << 20) || ((uintptr_t) dst & 3u))
        return ecb_check(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream), "host to device copy");
    const size_t need = (bytes + 255) & ~(size_t) 255;
    if (ctx->up_off + need > ctx->up_cap) {
        // everything staged so far must have been pulled before the region is reused (or replaced)
        ECB_CUDA(ctx, ecb_stream_sync(ctx));
        ctx->up_off = 0;
        if (need > ctx->up_cap) {
            if (ctx->up) cudaFreeHost(ctx->up);
            ctx->up = nullptr;
            ctx->up_cap = 0;
            const size_t cap = std::max(need * 2, (size_t) 2 << 20);
            ECB_CUDA(ctx, cudaHostAlloc(&ctx->up, cap, cudaHostAllocMapped));
            ctx->up_cap = cap;
        }
    }
    char *stage = (char *) ctx->up + ctx->up_off;
    ctx->up_off += need;
    memcpy(stage, src, bytes);
    void *dstage = nullptr;
    ECB_CUDA(ctx, cudaHostGetDevicePointer(&dstage, stage, 0));
    const size_t words = bytes >> 2;
    const int grid = (int) std::min<size_t>((words + 255) / 256 + 1, 128);
    k_pull<<<grid, 256, 0, ctx->stream>>>((uint32_t *) dst, (const uint32_t *) dstage, words, bytes);
    ECB_LAUNCHED(ctx);
    return ecb_check(ctx, cudaGetLastError(), "k_pull launch");
}

extern "C" {

const char *ecb_version(void) { return "eventcalib_b200 0.1 (sm_100a)"; }

int ecb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int ecb_ctx_create(int device, void *stream, ecb_ctx **out) {
    if (!out) return ECB_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) return ECB_ERR_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return ECB_ERR_CUDA;
    ecb_ctx *c = new ecb_ctx();
    c->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        delete c;
        return ECB_ERR_CUDA;
    }
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = (int) prop.sharedMemPerBlockOptin;
    if (stream) {
        c->stream = (cudaStream_t) stream;
    } else {
        if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete c;
            return ECB_ERR_CUDA;
        }
        c->own_stream = true;
    }
    if (const char *e = getenv("ECB_BLOCKING_SYNC"))
        if (atoi(e) > 0 && cudaEventCreateWithFlags(&c->sync_ev, (atoi(e) == 1 ? cudaEventBlockingSync : 0) | cudaEventDisableTiming) == cudaSuccess)
            c->sync_mode = atoi(e) == 1 ? 1 : 2;
    *out = c;
    return ECB_OK;
}

void ecb_cost_free(ecb_ctx *ctx);
void ecb_covariance_free(ecb_ctx *ctx);

void ecb_ctx_destroy(ecb_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    ecb_covariance_free(c);
    ecb_cost_free(c);
    DevBuf *bufs[] = {&c->ev_raw, &c->ev_t, &c->ev_xyp, &c->ev_flag, &c->win_t, &c->win_lohi, &c->win_ptoff, &c->summary,
                      &c->arrive, &c->pts[0], &c->pts[1], &c->labels[0], &c->labels[1], &c->scratch, &c->ktab, &c->kmem,
                      &c->cand, &c->status, &c->db_pix, &c->db_off, &c->db_labels, &c->db_hdr, &c->db_scratch, &c->db_dims,
                      &c->fit_in, &c->fit_off, &c->fit_out, &c->db_hdr_b, &c->db_ktab, &c->db_counter, &c->kd_tree, &c->bfs_key,
                      &c->bfs_items, &c->bfs_front, &c->bfs_tab, &c->ord_htab, &c->pair_tab, &c->pose_io,
                      &c->motion_io, &c->gyro_io};
    for (DevBuf *b : bufs)
        if (b->p) cudaFree(b->p);
    for (DevBuf &b : c->gh)
        if (b.p) cudaFree(b.p);
    for (int i = 0; i < ECB_N_STAGES; ++i)
        for (int j = 0; j < 2; ++j)
            if (c->pev[i][j]) cudaEventDestroy(c->pev[i][j]);
    if (c->sync_ev) cudaEventDestroy(c->sync_ev);
    if (c->pinned) cudaFreeHost(c->pinned);
    if (c->up) cudaFreeHost(c->up);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
}

const char *ecb_last_error(const ecb_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }
uint64_t ecb_launch_count(const ecb_ctx *ctx) { return ctx ? ctx->launches : 0; }

int ecb_synchronize(ecb_ctx *ctx) {
    if (!ctx) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    return ecb_check(ctx, ecb_stream_sync(ctx), "stream synchronize");
}

int ecb_set_profiling(ecb_ctx *ctx, int on) {
    if (!ctx) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    if (on && !ctx->pev[0][0])
        for (int i = 0; i < ECB_N_STAGES; ++i)
            for (int j = 0; j < 2; ++j) ECB_CUDA(ctx, cudaEventCreate(&ctx->pev[i][j]));
    ctx->prof = on != 0;
    for (int i = 0; i < ECB_N_STAGES; ++i) ctx->pev_used[i] = false;
    return ECB_OK;
}

int ecb_stage_ms(ecb_ctx *ctx, float *out) {
    if (!ctx || !out) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    ECB_CUDA(ctx, ecb_stream_sync(ctx));
    for (int i = 0; i < ECB_N_STAGES; ++i) {
        out[i] = 0.f;
        if (ctx->pev_used[i]) ECB_CUDA(ctx, cudaEventElapsedTime(&out[i], ctx->pev[i][0], ctx->pev[i][1]));
    }
    return ECB_OK;
}

int ecb_set_sensor(ecb_ctx *ctx, int width, int height) {
    if (!ctx) return ECB_ERR_ARG;
    if (width < 1 || height < 1 || width > 32767 || height > 32767 || (int64_t) width * height > (1 << 20))
        return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "sensor %dx%d outside the supported range (<= 2^20 pixels)", width, height);
    ctx->width = width;
    ctx->height = height;
    return ECB_OK;
}

int64_t ecb_num_events(const ecb_ctx *ctx) { return ctx ? ctx->n_events : 0; }

static int unpack_events(ecb_ctx *ctx, const void *d_raw, int64_t n) {
    int rc;
    ++ctx->events_gen;
    if ((rc = ecb_reserve(ctx, ctx->ev_t, (size_t) n * 8))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->ev_xyp, (size_t) n * 4))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->ev_flag, 16))) return rc;
    ECB_CUDA(ctx, cudaMemsetAsync(ctx->ev_flag.p, 0, 16, ctx->stream));
    if ((rc = ecb_launch_ingest(ctx, d_raw, n))) return rc;
    uint32_t flag = 0;
    if ((rc = ecb_d2h(ctx, &flag, ctx->ev_flag.p, 4))) return rc;
    ctx->n_events = n;
    if (flag & 1u) {
        ctx->n_events = 0;
        return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "event stream holds non-integer or out-of-sensor pixel coordinates");
    }
    // an unsorted file: the reference's multimap load orders it by stamp, file order among equal stamps
    // (eventCameraCalib.cpp:154-163) — a stable device radix sort here
    if ((flag & 2u) && (rc = ecb_sort_events_by_time(ctx, n))) {
        ctx->n_events = 0;
        return rc;
    }
    return ECB_OK;
}

int ecb_load_events_device(ecb_ctx *ctx, const void *d_records, int64_t n) {
    if (!ctx || (!d_records && n > 0) || n < 0) return ECB_ERR_ARG;
    if (ctx->width <= 0) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_set_sensor must be called before loading events");
    if (((uintptr_t) d_records & 15u) != 0) return ecb_fail(ctx, ECB_ERR_ARG, "device record buffer must be 16-byte aligned");
    cudaSetDevice(ctx->device);
    return unpack_events(ctx, d_records, n);
}

int ecb_load_events_host(ecb_ctx *ctx, const void *records, int64_t n) {
    if (!ctx || (!records && n > 0) || n < 0) return ECB_ERR_ARG;
    if (ctx->width <= 0) return ecb_fail(ctx, ECB_ERR_STATE, "ecb_set_sensor must be called before loading events");
    cudaSetDevice(ctx->device);
    int rc;
    if ((rc = ecb_reserve(ctx, ctx->ev_raw, (size_t) n * 25 + 16))) return rc;
    ECB_CUDA(ctx, cudaMemcpyAsync(ctx->ev_raw.p, records, (size_t) n * 25, cudaMemcpyHostToDevice, ctx->stream));
    return unpack_events(ctx, ctx->ev_raw.p, n);
}

// --------------------------------------------------------------------------------------- front end ----
static int fill_stencil(ecb_ctx *ctx, ClusterArgs &a, double eps) {
    if (!(eps >= 1.0) || eps > ECB_MAX_EPS)
        return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "dbscan eps %.3f outside the supported range [1, %d]", eps, ECB_MAX_EPS);
    a.E = (int) floor(eps);
    a.eps_int = (eps == floor(eps)) ? (int) eps : -1;
    for (int dy = 0; dy <= ECB_MAX_EPS; ++dy) {
        int w = -1;
        if (dy <= a.E) {
            // largest integer w with w*w + dy*dy <= eps*eps, evaluated like the reference: d2 <= SQ(range) in f64
            w = 0;
            while ((double) (w + 1) * (w + 1) + (double) dy * dy <= eps * eps) ++w;
        }
        a.halfw[dy] = (int8_t) w;
    }
    return ECB_OK;
}

int ecb_frontend_run(ecb_ctx *ctx, const double *windows, int n_win, const ecb_frontend_params *params) {
    if (!ctx || !params || (n_win > 0 && !windows) || n_win < 0) return ECB_ERR_ARG;
    if (ctx->n_events <= 0) return ecb_fail(ctx, ECB_ERR_STATE, "no events loaded");
    if (params->dbscan_min_pts < 1) return ecb_fail(ctx, ECB_FAILED, "min_pts < 1 (DBSCAN::Run returns FAILED)");
    if (params->order_mode != 0 && params->order_mode != 1)
        return ecb_fail(ctx, ECB_ERR_ARG, "order_mode %d unknown", params->order_mode);
    if (params->median_mode > 1) return ecb_fail(ctx, ECB_ERR_ARG, "median_mode %u unknown", params->median_mode);
    cudaSetDevice(ctx->device);
    int rc;
    ctx->fp = *params;
    ctx->n_win = 0;
    // kept-cluster table capacity per (window, polarity): fixed when the caller names one (overflow -> ECB_PB_CLUSTER_CAP),
    // else automatic — the cluster / pair stages are repeated with a larger table when a window overflows (the reference
    // has no cap, CirclesEventFrame.cpp:89-117), and the context remembers the capacity for the next run
    const bool auto_k = params->max_clusters == 0;
    int max_k = auto_k ? ctx->max_k_auto : (int) std::min<uint32_t>(params->max_clusters, 1u << 20);
    ClusterArgs ca;
    memset(&ca, 0, sizeof ca);
    if ((rc = fill_stencil(ctx, ca, params->dbscan_eps))) return rc;
    if (n_win == 0) return ECB_OK;

    // window bounds
    if ((rc = ecb_reserve(ctx, ctx->win_t, (size_t) n_win * 16))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->win_lohi, (size_t) n_win * 16))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->win_ptoff, (size_t) n_win * 8))) return rc;
    if ((rc = ecb_h2d(ctx, ctx->win_t.p, windows, (size_t) n_win * 16))) return rc;
    if ((rc = ecb_launch_bounds(ctx, (const double *) ctx->win_t.p, n_win, (int64_t *) ctx->win_lohi.p))) return rc;
    ctx->h_lohi.resize((size_t) 2 * n_win);
    ctx->h_ptoff.resize((size_t) n_win);
    if ((rc = ecb_d2h(ctx, ctx->h_lohi.data(), ctx->win_lohi.p, (size_t) n_win * 16))) return rc;
    int64_t total = 0, max_cnt = 0;
    for (int w = 0; w < n_win; ++w) {
        int64_t cnt = std::max<int64_t>(0, ctx->h_lohi[2 * w + 1] - ctx->h_lohi[2 * w]);
        ctx->h_ptoff[w] = total;
        total += cnt;
        max_cnt = std::max(max_cnt, cnt);
    }
    if (max_cnt > 0x3FFFFFFF) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "window with %lld events", (long long) max_cnt);
    ctx->total_points = total;
    if ((rc = ecb_h2d(ctx, ctx->win_ptoff.p, ctx->h_ptoff.data(), (size_t) n_win * 8))) return rc;

    const size_t slots = (size_t) std::max<int64_t>(total, 1);
    if ((rc = ecb_reserve(ctx, ctx->arrive, 2 * slots * 4))) return rc;
    for (int p = 0; p < 2; ++p) {
        if ((rc = ecb_reserve(ctx, ctx->pts[p], slots * 4))) return rc;
        if ((rc = ecb_reserve(ctx, ctx->labels[p], slots * 4))) return rc;
    }
    if ((rc = ecb_reserve(ctx, ctx->kmem, 2 * slots * 4))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->db_dims, (size_t) 2 * n_win * sizeof(ProbDesc)))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->db_hdr, (size_t) 2 * n_win * sizeof(ProbHdr)))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->summary, (size_t) n_win * sizeof(ecb_window_summary)))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->status, 64))) return rc;

    WindowArgs wa;
    wa.xyp = (const uint32_t *) ctx->ev_xyp.p;
    wa.lohi = (const int64_t *) ctx->win_lohi.p;
    wa.ptoff = (const int64_t *) ctx->win_ptoff.p;
    wa.arrive[0] = (uint32_t *) ctx->arrive.p;
    wa.arrive[1] = (uint32_t *) ctx->arrive.p + slots;
    wa.pts[0] = (uint32_t *) ctx->pts[0].p;
    wa.pts[1] = (uint32_t *) ctx->pts[1].p;
    wa.prob = (ProbDesc *) ctx->db_dims.p;
    wa.n_win = n_win;
    wa.W = ctx->width;
    wa.H = ctx->height;
    wa.max_n = (uint32_t *) ctx->status.p + 4;
    wa.order_mode = params->order_mode;
    ECB_CUDA(ctx, cudaMemsetAsync(ctx->status.p, 0, 64, ctx->stream));
    if ((rc = ecb_launch_window(ctx, wa))) return rc;
    uint32_t max_nm[2] = {0, 0};
    if ((rc = ecb_d2h(ctx, max_nm, wa.max_n, 8))) return rc;
    const uint32_t max_n = max_nm[0];
    if (params->order_mode == 1) {  // pid order = iteration order of the reference's unordered_sets
        OrderArgs oa;
        memset(&oa, 0, sizeof oa);
        oa.prob = (const ProbDesc *) ctx->db_dims.p;
        oa.n_prob = 2 * n_win;
        oa.work_counter = (unsigned *) ctx->status.p;
        for (int p = 0; p < 2; ++p) {
            oa.arrive[p] = wa.arrive[p];
            oa.pts[p] = wa.pts[p];
        }
        if ((rc = ecb_launch_order(ctx, oa, (int) max_nm[1]))) return rc;
    }

  for (int attempt = 0;; ++attempt) {  // repeated (rarely) with a larger kept-cluster table in the automatic mode
    if ((rc = ecb_reserve(ctx, ctx->ktab, (size_t) 2 * n_win * max_k * sizeof(KeptCluster)))) return rc;
    ctx->cand_stride = max_k;
    if ((rc = ecb_reserve(ctx, ctx->cand, (size_t) n_win * ctx->cand_stride * 5 * 8))) return rc;
    uint32_t *const d_max_kept = (uint32_t *) ctx->status.p + 12;
    ca.max_kept = d_max_kept;
    ca.prob = (const ProbDesc *) ctx->db_dims.p;
    ca.n_prob = 2 * n_win;
    ca.work_counter = (unsigned *) ctx->status.p;
    for (int p = 0; p < 2; ++p) {
        ca.pix[p] = (const uint32_t *) ctx->pts[p].p;
        ca.labels[p] = (int32_t *) ctx->labels[p].p;
        ca.kmem[p] = (uint32_t *) ctx->kmem.p + p * slots;
    }
    ca.hdr = (ProbHdr *) ctx->db_hdr.p;
    ca.ktab = (KeptCluster *) ctx->ktab.p;
    ca.max_k = max_k;
    ca.W = ctx->width;
    ca.H = ctx->height;
    ca.PW = ecb_cluster_row_words(ca.W, ca.E);
    ca.PH = ca.H + 2 * ca.E;
    ca.min_pts = params->dbscan_min_pts;
    ca.cluster_min = params->cluster_min;
    const bool exact = params->median_mode == 1;
    int bfs_cap = 0;
    if (exact) {  // reference-exact medians: export the kd-tree, queue the clusters whose median norm is tied
        bfs_cap = (int) std::min<size_t>((size_t) 2 * n_win * max_k, 2 * slots / std::max<uint32_t>(params->cluster_min, 1u) + 16);
        if ((rc = ecb_reserve(ctx, ctx->kd_tree, 8 * slots * 4))) return rc;
        if ((rc = ecb_reserve(ctx, ctx->bfs_key, 2 * slots * 8))) return rc;
        if ((rc = ecb_reserve(ctx, ctx->bfs_items, (size_t) bfs_cap * sizeof(BfsItem) + 16))) return rc;
        ca.exact_order = 1;
        for (int p = 0; p < 2; ++p) ca.kd_nodes[p] = (uint32_t *) ctx->kd_tree.p + (size_t) (4 * p) * slots;
        ca.bfs_items = (BfsItem *) ((char *) ctx->bfs_items.p + 16);
        ca.bfs_count = (unsigned *) ctx->bfs_items.p;
        ca.bfs_cap = bfs_cap;
        ECB_CUDA(ctx, cudaMemsetAsync(ctx->bfs_items.p, 0, 16, ctx->stream));
    }
    if ((rc = ecb_launch_cluster(ctx, ca, (int) max_n))) return rc;
    if (exact) {
        BfsArgs ba;
        memset(&ba, 0, sizeof ba);
        ba.items = ca.bfs_items;
        ba.count = ca.bfs_count;
        ba.max_items = bfs_cap;
        ba.prob = ca.prob;
        for (int p = 0; p < 2; ++p) {
            ba.pix[p] = ca.pix[p];
            ba.labels[p] = ca.labels[p];
            ba.kd_nodes[p] = (const uint4 *) ca.kd_nodes[p];
            ba.members[p] = ca.kmem[p];
            ba.scratch[p] = wa.arrive[p];  // the arrival lists are dead by now
            ba.key[p] = (unsigned long long *) ctx->bfs_key.p + (size_t) p * slots;
        }
        ba.init_keys = 1;
        ba.ktab = ca.ktab;
        ba.max_k = max_k;
        ba.eps = params->dbscan_eps;
        if ((rc = ecb_launch_bfs(ctx, ba))) return rc;
    }

    PairArgs pa;
    pa.prob = ca.prob;
    pa.hdr = ca.hdr;
    pa.ktab = ca.ktab;
    for (int p = 0; p < 2; ++p) {
        pa.pts[p] = ca.pix[p];
        pa.kmem[p] = ca.kmem[p];
    }
    pa.lohi = wa.lohi;
    pa.summary = (ecb_window_summary *) ctx->summary.p;
    pa.cand = (double *) ctx->cand.p;
    pa.n_win = n_win;
    pa.max_k = max_k;
    pa.cand_stride = ctx->cand_stride;
    pa.smem_cap = (int) max_n;
    pa.fit_circle = params->fit_circle;
    pa.knn_num = params->knn_num < 1 ? 1 : params->knn_num;
    pa.rows_cols = params->rows_cols;
    pa.rthr = params->radius_threshold;
    {   // word 8 of the status block (zeroed at the start of this run) = k_pair's window counter
        static const int pair_dyn = getenv("ECB_PAIR_DYN") ? atoi(getenv("ECB_PAIR_DYN")) : 1;
        pa.win_counter = pair_dyn ? (unsigned *) ctx->status.p + 8 : nullptr;
    }
    if ((rc = ecb_launch_pair(ctx, pa))) return rc;
    if (!auto_k) break;
    uint32_t max_kept = 0;
    if ((rc = ecb_d2h(ctx, &max_kept, d_max_kept, 4))) return rc;
    if (max_kept <= (uint32_t) max_k) break;
    if (attempt >= 2) return ecb_fail(ctx, ECB_ERR_STATE, "kept-cluster table still too small after resizing (%u > %d)", max_kept, max_k);
    max_k = (int) ((max_kept + 63u) & ~63u);
    ctx->max_k_auto = max_k;
    ECB_CUDA(ctx, cudaMemsetAsync((uint32_t *) ctx->status.p + 8, 0, 32, ctx->stream));  // pair window counter, max_kept
  }
    ctx->n_win = n_win;
    return ECB_OK;
}

int ecb_frontend_summary(ecb_ctx *ctx, ecb_window_summary *out, int n_win) {
    if (!ctx || !out) return ECB_ERR_ARG;
    if (n_win > ctx->n_win) n_win = ctx->n_win;
    cudaSetDevice(ctx->device);
    return ecb_d2h(ctx, out, ctx->summary.p, (size_t) n_win * sizeof(ecb_window_summary));
}

int64_t ecb_frontend_total_points(ecb_ctx *ctx, int polarity) {
    (void) polarity;
    return ctx ? ctx->total_points : 0;
}

int ecb_frontend_points(ecb_ctx *ctx, int polarity, double *xy, int32_t *labels) {
    if (!ctx || polarity < 0 || polarity > 1) return ECB_ERR_ARG;
    if (ctx->n_win <= 0) return ecb_fail(ctx, ECB_ERR_STATE, "no front-end results");
    cudaSetDevice(ctx->device);
    const size_t slots = (size_t) ctx->total_points;
    if (labels)
        ECB_CUDA(ctx, cudaMemcpyAsync(labels, ctx->labels[polarity].p, slots * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (xy) {
        std::vector<uint32_t> pix(slots);
        ECB_CUDA(ctx, cudaMemcpyAsync(pix.data(), ctx->pts[polarity].p, slots * 4, cudaMemcpyDeviceToHost, ctx->stream));
        ECB_CUDA(ctx, ecb_stream_sync(ctx));
        for (size_t i = 0; i < slots; ++i) {
            xy[2 * i] = (double) ECB_PIX_X(pix[i]);
            xy[2 * i + 1] = (double) ECB_PIX_Y(pix[i]);
        }
    }
    return ecb_check(ctx, ecb_stream_sync(ctx), "points copy");
}

int ecb_frontend_candidates(ecb_ctx *ctx, double *out, int max_cand) {
    if (!ctx || !out || max_cand < 1) return ECB_ERR_ARG;
    if (ctx->n_win <= 0) return ecb_fail(ctx, ECB_ERR_STATE, "no front-end results");
    cudaSetDevice(ctx->device);
    const int k = std::min(max_cand, ctx->cand_stride);
    const size_t bytes = (size_t) ctx->n_win * k * 40;
    int rc = reserve_pinned(ctx, bytes);
    if (rc) return rc;
    ECB_CUDA(ctx, cudaMemcpy2DAsync(ctx->pinned, (size_t) k * 40, ctx->cand.p, (size_t) ctx->cand_stride * 40, (size_t) k * 40,
                                    (size_t) ctx->n_win, cudaMemcpyDeviceToHost, ctx->stream));
    ECB_CUDA(ctx, ecb_stream_sync(ctx));
    for (int w = 0; w < ctx->n_win; ++w)
        memcpy(out + (size_t) w * max_cand * 5, (const char *) ctx->pinned + (size_t) w * k * 40, (size_t) k * 40);
    return ECB_OK;
}

int ecb_frontend_clusters(ecb_ctx *ctx, int window, int polarity, int32_t *raw_id, int32_t *size, int32_t *median_pid,
                          int cap) {
    if (!ctx || window < 0 || window >= ctx->n_win || polarity < 0 || polarity > 1) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    const int max_k = ctx->cand_stride;
    std::vector<KeptCluster> k((size_t) max_k);
    ProbHdr h;
    const size_t pb = (size_t) 2 * window + polarity;
    ECB_CUDA(ctx, cudaMemcpyAsync(&h, (ProbHdr *) ctx->db_hdr.p + pb, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    ECB_CUDA(ctx, cudaMemcpyAsync(k.data(), (KeptCluster *) ctx->ktab.p + pb * max_k, sizeof(KeptCluster) * max_k,
                                  cudaMemcpyDeviceToHost, ctx->stream));
    ECB_CUDA(ctx, ecb_stream_sync(ctx));
    int n = std::min(h.n_kept, cap);
    for (int i = 0; i < n; ++i) {
        if (raw_id) raw_id[i] = k[i].raw_id;
        if (size) size[i] = k[i].size;
        if (median_pid) median_pid[i] = k[i].med_pid;
    }
    return n;
}

int ecb_frontend_rectify(ecb_ctx *ctx, const int32_t *window_index, int n_frames, int n_circles,
                         const double *image_points, double inlier_threshold, int rows, int cols, int asymmetric,
                         double *out, int32_t *frame_ok) {
    if (!ctx || n_frames < 0 || n_circles < 1 || (n_frames > 0 && (!window_index || !image_points || !out))) return ECB_ERR_ARG;
    if (ctx->n_win <= 0) return ecb_fail(ctx, ECB_ERR_STATE, "no front-end results");
    if (n_frames == 0) return ECB_OK;
    for (int i = 0; i < n_frames; ++i)
        if (window_index[i] < 0 || window_index[i] >= ctx->n_win)
            return ecb_fail(ctx, ECB_ERR_ARG, "frame %d: window index %d outside the last run's %d windows", i, window_index[i], ctx->n_win);
    cudaSetDevice(ctx->device);
    int rc;
    const size_t items = (size_t) n_frames * n_circles;
    if ((rc = ecb_reserve(ctx, ctx->fit_in, items * 80 + (size_t) n_frames * 4 + 16))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->fit_out, items * 24))) return rc;
    double *d_img = (double *) ctx->fit_in.p;
    int32_t *d_win = (int32_t *) (d_img + items * 10);
    if ((rc = ecb_h2d(ctx, d_img, image_points, items * 80))) return rc;
    if ((rc = ecb_h2d(ctx, d_win, window_index, (size_t) n_frames * 4))) return rc;
    PairArgs pa;
    memset(&pa, 0, sizeof pa);
    pa.prob = (const ProbDesc *) ctx->db_dims.p;
    pa.hdr = (const ProbHdr *) ctx->db_hdr.p;
    pa.ktab = (const KeptCluster *) ctx->ktab.p;
    const int32_t *labels[2];
    for (int p = 0; p < 2; ++p) {
        pa.pts[p] = (const uint32_t *) ctx->pts[p].p;
        labels[p] = (const int32_t *) ctx->labels[p].p;
    }
    pa.max_k = ctx->cand_stride;
    if ((rc = ecb_launch_rectify(ctx, d_win, n_frames, n_circles, d_img, (double *) ctx->fit_out.p, pa, labels, inlier_threshold)))
        return rc;
    if ((rc = ecb_d2h(ctx, out, ctx->fit_out.p, items * 24))) return rc;
    if (frame_ok) {  // :585-609 (host: a few dozen integer operations per frame)
        auto on_edge = [&](int e, int i) -> bool {
            const int step = (asymmetric ? 2 : 1) * cols;
            if (e == 0) return i < cols;
            if (e == 1) return i >= (rows - 1) * cols && i < rows * cols;
            if (e == 2) return i < rows * cols && i % step == 0;
            const int first = asymmetric ? 2 * cols - 1 : cols - 1;
            return i >= first && i < rows * cols && (i - first) % step == 0;
        };
        int size_[4] = {0, 0, 0, 0};
        for (int e = 0; e < 4; ++e)
            for (int i = 0; i < rows * cols; ++i) size_[e] += on_edge(e, i);
        for (int f = 0; f < n_frames; ++f) {
            int score[4] = {0, 0, 0, 0}, counter = 0;
            for (int i = 0; i < n_circles; ++i)
                if (out[((size_t) f * n_circles + i) * 3 + 2] < 0) {
                    for (int e = 0; e < 4; ++e) score[e] += on_edge(e, i);
                    ++counter;
                }
            int okf = 1;
            if (!ctx->fp.fit_circle)
                for (int e = 0; e < 4; ++e)
                    if (score[e] >= size_[e] - 1) okf = 0;
            if (counter >= 0.2 * (cols * rows)) okf = 0;
            frame_ok[f] = okf;
        }
    }
    return ECB_OK;
}

int ecb_frontend_device_ptrs(ecb_ctx *ctx, void **d_summary, void **d_candidates, int *cand_stride) {
    if (!ctx) return ECB_ERR_ARG;
    if (d_summary) *d_summary = ctx->summary.p;
    if (d_candidates) *d_candidates = ctx->cand.p;
    if (cand_stride) *cand_stride = ctx->cand_stride;
    return ECB_OK;
}

// ------------------------------------------------------------------------- DBSCAN::Run boundary ----
static int dbscan_batch(ecb_ctx *ctx, const double *xy, const int64_t *offsets, int n_problems, double eps,
                        uint32_t min_pts, int32_t *labels, int32_t *n_clusters, uint32_t *status, int32_t *cluster_sizes,
                        uint32_t *members) {
    if (!ctx || !offsets || n_problems < 0 || (!xy && n_problems > 0)) return ECB_ERR_ARG;
    const bool ordered = cluster_sizes && members;
    if (min_pts < 1) return ecb_fail(ctx, ECB_FAILED, "min < 1 (dbscan.h:123)");
    cudaSetDevice(ctx->device);
    int rc;
    ClusterArgs ca;
    memset(&ca, 0, sizeof ca);
    if (n_problems == 0) return ECB_OK;
    // Inputs outside the bitmap kernel's domain (distinct integer pixels, 1 <= eps <= 15, bounded extent) take the general
    // grid-hash path (ecb_gridhash.cu) — same results as the reference on everything it accepts (dbscan.h:40,70,115-177).
    auto general = [&]() {
        if (status)
            for (int k = 0; k < n_problems; ++k) status[k] = 0;
        return ecb_dbscan_general(ctx, xy, 2, offsets, n_problems, eps, min_pts, labels, n_clusters, cluster_sizes, members);
    };
    if (!(eps >= 1.0) || eps > ECB_MAX_EPS) return general();
    if ((rc = fill_stencil(ctx, ca, eps))) return rc;
    const int64_t total = offsets[n_problems];
    // host-side packing: integer check, bounding boxes (the window path does this on the device in k_ingest)
    std::vector<uint32_t> pix((size_t) std::max<int64_t>(total, 1));
    std::vector<ProbDesc> pd((size_t) n_problems);
    int Wmax = 1, Hmax = 1, max_n = 0;
    for (int k = 0; k < n_problems; ++k) {
        const int64_t b = offsets[k], e = offsets[k + 1];
        if (e - b < 1) return ecb_fail(ctx, ECB_FAILED, "problem %d: V->size() < 1 (dbscan.h:121)", k);
        if (e - b > 0x3FFFFFFF) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "problem %d too large", k);
        int xmin = 1 << 30, ymin = 1 << 30, xmax = -1, ymax = -1;
        for (int64_t i = b; i < e; ++i) {
            const double x = xy[2 * i], y = xy[2 * i + 1];
            const int xi = (int) x, yi = (int) y;
            if (!(x >= 0.0 && x < 32768.0 && y >= 0.0 && y < 32768.0 && (double) xi == x && (double) yi == y)) return general();
            pix[(size_t) i] = (uint32_t) xi | ((uint32_t) yi << 15);
            xmin = std::min(xmin, xi);
            ymin = std::min(ymin, yi);
            xmax = std::max(xmax, xi);
            ymax = std::max(ymax, yi);
        }
        ProbDesc d;
        memset(&d, 0, sizeof d);
        d.off = b;
        d.n = (int32_t) (e - b);
        d.pol = 0;
        d.x0 = xmin;
        d.y0 = ymin;
        pd[(size_t) k] = d;
        Wmax = std::max(Wmax, xmax - xmin + 1);
        Hmax = std::max(Hmax, ymax - ymin + 1);
        max_n = std::max(max_n, d.n);
    }
    if ((int64_t) (Wmax + 2 * ca.E + 64) * (Hmax + 2 * ca.E) > (1ll << 21)) return general();  // bit planes beyond 256 KB
    const size_t slots = (size_t) std::max<int64_t>(total, 1);
    const int max_k = 1;  // no kept-cluster tables on this path (cluster_min below)
    if ((rc = ecb_reserve(ctx, ctx->db_pix, slots * 4))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->db_labels, slots * 4))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->db_scratch, slots * 4))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->db_off, (size_t) n_problems * sizeof(ProbDesc)))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->db_hdr_b, (size_t) n_problems * sizeof(ProbHdr)))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->db_ktab, (size_t) n_problems * max_k * sizeof(KeptCluster)))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->db_counter, 64))) return rc;
    ECB_CUDA(ctx, cudaMemcpyAsync(ctx->db_pix.p, pix.data(), slots * 4, cudaMemcpyHostToDevice, ctx->stream));
    ECB_CUDA(ctx, cudaMemcpyAsync(ctx->db_off.p, pd.data(), (size_t) n_problems * sizeof(ProbDesc), cudaMemcpyHostToDevice,
                                  ctx->stream));
    ca.prob = (const ProbDesc *) ctx->db_off.p;
    ca.n_prob = n_problems;
    ca.work_counter = (unsigned *) ctx->db_counter.p;
    ca.pix[0] = ca.pix[1] = (const uint32_t *) ctx->db_pix.p;
    ca.labels[0] = ca.labels[1] = (int32_t *) ctx->db_labels.p;
    ca.kmem[0] = ca.kmem[1] = (uint32_t *) ctx->db_scratch.p;
    ca.hdr = (ProbHdr *) ctx->db_hdr_b.p;
    ca.ktab = (KeptCluster *) ctx->db_ktab.p;
    ca.max_k = max_k;
    ca.W = Wmax;
    ca.H = Hmax;
    ca.PW = ecb_cluster_row_words(ca.W, ca.E);
    ca.PH = ca.H + 2 * ca.E;
    ca.min_pts = min_pts;
    ca.cluster_min = 0x7FFFFFFF;  // no kept-cluster tables on this path
    ca.max_kept = nullptr;
    if (ordered) {
        if ((rc = ecb_reserve(ctx, ctx->kd_tree, 4 * slots * 4))) return rc;
        ca.exact_order = 1;
        ca.kd_nodes[0] = ca.kd_nodes[1] = (uint32_t *) ctx->kd_tree.p;
        ca.bfs_count = (unsigned *) ctx->db_counter.p + 4;  // unused by k_cluster here (no kept clusters), must be valid
        ca.bfs_cap = 0;
    }
    if ((rc = ecb_launch_cluster(ctx, ca, max_n))) return rc;
    if (ordered) {
        // every cluster -> one work item; member lists of problem k at members[offsets[k] + offset of the cluster]
        if ((rc = ecb_reserve(ctx, ctx->bfs_key, slots * 8))) return rc;
        if ((rc = ecb_reserve(ctx, ctx->bfs_items, slots * sizeof(BfsItem) + 16))) return rc;
        if ((rc = ecb_reserve(ctx, ctx->bfs_front, slots * 4))) return rc;
        if ((rc = ecb_reserve(ctx, ctx->bfs_tab, 3 * slots * 4))) return rc;
        ECB_CUDA(ctx, cudaMemsetAsync(ctx->bfs_key.p, 0xFF, slots * 8, ctx->stream));
        ECB_CUDA(ctx, cudaMemsetAsync(ctx->bfs_items.p, 0, 16, ctx->stream));
        uint32_t *csize = (uint32_t *) ctx->bfs_tab.p, *cseed = csize + slots, *coff = cseed + slots;
        BfsItem *items = (BfsItem *) ((char *) ctx->bfs_items.p + 16);
        if ((rc = ecb_launch_bfs_all_items(ctx, ca.prob, ca.hdr, n_problems, ca.labels[0], csize, cseed, coff, items,
                                           (unsigned *) ctx->bfs_items.p, (int) slots)))
            return rc;
        BfsArgs ba;
        memset(&ba, 0, sizeof ba);
        ba.items = items;
        ba.count = (const unsigned *) ctx->bfs_items.p;
        ba.max_items = (int) slots;
        ba.prob = ca.prob;
        for (int p = 0; p < 2; ++p) {
            ba.pix[p] = ca.pix[0];
            ba.labels[p] = ca.labels[0];
            ba.kd_nodes[p] = (const uint4 *) ca.kd_nodes[0];
            ba.members[p] = (uint32_t *) ctx->db_scratch.p;
            ba.scratch[p] = (uint32_t *) ctx->bfs_front.p;
            ba.key[p] = (unsigned long long *) ctx->bfs_key.p;
        }
        ba.init_keys = 0;
        ba.eps = eps;
        if ((rc = ecb_launch_bfs(ctx, ba))) return rc;
        ECB_CUDA(ctx, cudaMemcpyAsync(members, ctx->db_scratch.p, (size_t) total * 4, cudaMemcpyDeviceToHost, ctx->stream));
        ECB_CUDA(ctx, cudaMemcpyAsync(cluster_sizes, csize, (size_t) total * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    std::vector<ProbHdr> hdr((size_t) n_problems);
    if (labels) ECB_CUDA(ctx, cudaMemcpyAsync(labels, ctx->db_labels.p, (size_t) total * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ECB_CUDA(ctx, cudaMemcpyAsync(hdr.data(), ctx->db_hdr_b.p, (size_t) n_problems * sizeof(ProbHdr), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    ECB_CUDA(ctx, ecb_stream_sync(ctx));
    for (int k = 0; k < n_problems; ++k) {
        if (n_clusters) n_clusters[k] = hdr[(size_t) k].n_clusters;
        if (status) status[k] = hdr[(size_t) k].status;
        // duplicate points are distinct pids and neighbours of each other in the reference (dbscan.h:218): the bitmap cannot
        // hold them, the general path can
        if (hdr[(size_t) k].status & ECB_PB_DUPLICATE) return general();
    }
    return ECB_OK;
}

int ecb_dbscan_run_batch(ecb_ctx *ctx, const double *xy, const int64_t *offsets, int n_problems, double eps,
                         uint32_t min_pts, int32_t *labels, int32_t *n_clusters, uint32_t *status) {
    return dbscan_batch(ctx, xy, offsets, n_problems, eps, min_pts, labels, n_clusters, status, nullptr, nullptr);
}

int ecb_dbscan_run_batch_ordered(ecb_ctx *ctx, const double *xy, const int64_t *offsets, int n_problems, double eps,
                                 uint32_t min_pts, int32_t *labels, int32_t *n_clusters, uint32_t *status,
                                 int32_t *cluster_sizes, uint32_t *members) {
    if (!cluster_sizes || !members) return ECB_ERR_ARG;
    return dbscan_batch(ctx, xy, offsets, n_problems, eps, min_pts, labels, n_clusters, status, cluster_sizes, members);
}

int ecb_dbscan_run_ordered(ecb_ctx *ctx, const double *xy, int n, double eps, uint32_t min_pts, int32_t *labels,
                           int32_t *n_clusters, int32_t *cluster_sizes, uint32_t *members) {
    if (!ctx || !cluster_sizes || !members) return ECB_ERR_ARG;
    if (n < 1 || min_pts < 1) return ECB_FAILED;  // dbscan.h:121-123
    const int64_t off[2] = {0, n};
    return dbscan_batch(ctx, xy, off, 1, eps, min_pts, labels, n_clusters, nullptr, cluster_sizes, members);
}

int ecb_dbscan_run_nd(ecb_ctx *ctx, const double *pts, int n, int dim, double eps, uint32_t min_pts, int32_t *labels,
                      int32_t *n_clusters, int32_t *cluster_sizes, uint32_t *members) {
    if (!ctx || (!pts && n > 0) || ((cluster_sizes == nullptr) != (members == nullptr))) return ECB_ERR_ARG;
    if (n < 1 || dim < 1 || min_pts < 1) return ECB_FAILED;  // dbscan.h:121-123
    const int64_t off[2] = {0, n};
    if (dim == 2) return dbscan_batch(ctx, pts, off, 1, eps, min_pts, labels, n_clusters, nullptr, cluster_sizes, members);
    cudaSetDevice(ctx->device);
    return ecb_dbscan_general(ctx, pts, dim, off, 1, eps, min_pts, labels, n_clusters, cluster_sizes, members);
}

int ecb_dbscan_run(ecb_ctx *ctx, const double *xy, int n, double eps, uint32_t min_pts, int32_t *labels,
                   int32_t *n_clusters) {
    if (!ctx) return ECB_ERR_ARG;
    if (n < 1 || min_pts < 1) return ECB_FAILED;  // dbscan.h:121-123
    const int64_t off[2] = {0, n};
    return ecb_dbscan_run_batch(ctx, xy, off, 1, eps, min_pts, labels, n_clusters, nullptr);
}

// ----------------------------------------------------------------------------------- circle fit ----
int ecb_fit_circles(ecb_ctx *ctx, const double *xy, const int64_t *offsets, int n_sets, double *out) {
    if (!ctx || !xy || !offsets || !out || n_sets < 0) return ECB_ERR_ARG;
    if (n_sets == 0) return ECB_OK;
    cudaSetDevice(ctx->device);
    int rc;
    const int64_t total = offsets[n_sets];
    if ((rc = ecb_reserve(ctx, ctx->fit_in, (size_t) std::max<int64_t>(total, 1) * 16))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->fit_off, (size_t) (n_sets + 1) * 8))) return rc;
    if ((rc = ecb_reserve(ctx, ctx->fit_out, (size_t) n_sets * 24))) return rc;
    ECB_CUDA(ctx, cudaMemcpyAsync(ctx->fit_in.p, xy, (size_t) total * 16, cudaMemcpyHostToDevice, ctx->stream));
    ECB_CUDA(ctx, cudaMemcpyAsync(ctx->fit_off.p, offsets, (size_t) (n_sets + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = ecb_launch_fit(ctx, (const double *) ctx->fit_in.p, (const int64_t *) ctx->fit_off.p, n_sets,
                             (double *) ctx->fit_out.p)))
        return rc;
    ECB_CUDA(ctx, cudaMemcpyAsync(out, ctx->fit_out.p, (size_t) n_sets * 24, cudaMemcpyDeviceToHost, ctx->stream));
    return ecb_check(ctx, ecb_stream_sync(ctx), "fit copy");
}

// ---- receive buffers of the multi-GPU exchange ----
int ecb_device_alloc(ecb_ctx *ctx, size_t bytes, void **d_ptr) {
    if (!ctx || !d_ptr || bytes == 0) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    ECB_CUDA(ctx, cudaMalloc(d_ptr, bytes));
    ECB_CUDA(ctx, cudaMemset(*d_ptr, 0, bytes));
    return ECB_OK;
}

int ecb_device_free(ecb_ctx *ctx, void *d_ptr) {
    if (!ctx) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    return ecb_check(ctx, cudaFree(d_ptr), "cudaFree");
}

int ecb_ipc_export(ecb_ctx *ctx, void *d_ptr, void *handle64) {
    if (!ctx || !d_ptr || !handle64) return ECB_ERR_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    cudaSetDevice(ctx->device);
    cudaIpcMemHandle_t h;
    ECB_CUDA(ctx, cudaIpcGetMemHandle(&h, d_ptr));
    memcpy(handle64, &h, 64);
    return ECB_OK;
}

int ecb_ipc_open(ecb_ctx *ctx, const void *handle64, void **d_ptr) {
    if (!ctx || !d_ptr || !handle64) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    return ecb_check(ctx, cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle");
}

int ecb_enable_peer_access(ecb_ctx *ctx, int peer_device) {
    if (!ctx || peer_device < 0) return ECB_ERR_ARG;
    if (peer_device == ctx->device) return ECB_OK;
    cudaSetDevice(ctx->device);
    int can = 0;
    ECB_CUDA(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, peer_device));
    if (!can) return ecb_fail(ctx, ECB_ERR_UNSUPPORTED, "device %d cannot access device %d's memory", ctx->device, peer_device);
    const cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        return ECB_OK;
    }
    return ecb_check(ctx, e, "cudaDeviceEnablePeerAccess");
}

int ecb_ipc_close(ecb_ctx *ctx, void *d_ptr) {
    if (!ctx) return ECB_ERR_ARG;
    cudaSetDevice(ctx->device);
    return ecb_check(ctx, cudaIpcCloseMemHandle(d_ptr), "cudaIpcCloseMemHandle");
}

}  // extern "C"
