// b2n_ctx.cu -- context lifetime, model registry, resident bound, batched model
// evaluation.  Part of libb200nest.so (C ABI in include/b200nest.h).
#include "b2n_device.cuh"
#include <algorithm>
#include <time.h>
#include <map>
#include <mutex>

static std::mutex g_smem_mu;
static std::map<std::pair<int, const void*>, size_t> g_smem_limit;

int b2n_func_smem(b2n_ctx* ctx, const void* func, size_t bytes) {
    if (bytes <= 48 * 1024) return B2N_OK;                      // the default limit needs no opt-in
    std::lock_guard<std::mutex> lk(g_smem_mu);
    size_t& cur = g_smem_limit[std::make_pair(ctx->device, func)];
    if (bytes <= cur) return B2N_OK;
    B2N_CUDA(ctx, cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    cur = bytes;
    return B2N_OK;
}

extern "C" {

const char* b2n_version(void) { return "b200nest 0.1 (sm_100a)"; }

const char* b2n_strerror(int s) {
    switch (s) {
        case B2N_OK: return "ok";
        case B2N_ERR_CUDA: return "CUDA runtime error";
        case B2N_ERR_ARG: return "invalid argument";
        case B2N_ERR_SINGLE_POINT: return "Cannot compute a bounding ellipsoid of a single point.";
        case B2N_ERR_SINGULAR: return "The input precision matrix defining the ellipsoid is apparently singular";
        case B2N_ERR_ELL_INIT: return "Failed to initialize the ellipsoid to contain all the points";
        case B2N_ERR_INVALID_REGION: return "Rejecting invalid MultiEllipsoid region";
        case B2N_ERR_Q0: return "Ellipsoid check failed q=0";
        case B2N_ERR_SLICE_FAIL: return "Slice sampler has failed to find a valid point.";
        case B2N_ERR_NOMEM: return "out of memory";
        case B2N_ERR_UNSUPPORTED: return "unsupported configuration";
        case B2N_ERR_TOO_MANY_ELLS: return "max_ells too small";
        case B2N_ERR_PEER: return "peer exchange failed";
        case B2N_ERR_PLATEAU: return "No live points are above loglstar. Do you have a likelihood plateau ?";
        default: return "unknown status";
    }
}

const char* b2n_last_error(b2n_ctx* ctx) { return ctx ? ctx->err : "null ctx"; }

int b2n_init(int device, b2n_ctx** out) {
    if (!out) return B2N_ERR_ARG;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0 || device < 0 || device >= count) return B2N_ERR_CUDA;
    if (cudaSetDevice(device) != cudaSuccess) return B2N_ERR_CUDA;
    if (const char* e = getenv("B2N_BLOCKING_SYNC")) {          // many contexts driven by many host threads (replicas): waiting
        if (e[0] == '1') { cudaSetDeviceFlags(cudaDeviceScheduleBlockingSync); cudaGetLastError(); }   // threads sleep instead of spinning
    }
    b2n_ctx* ctx = new b2n_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return B2N_ERR_CUDA; }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
        delete ctx;
        return B2N_ERR_CUDA;
    }
    ctx->own_stream = true;
    {   // (a failure here only costs the priority)
        int lo = 0, hi = 0;
        if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess ||
            cudaStreamCreateWithPriority(&ctx->stream_hi, cudaStreamNonBlocking, hi) != cudaSuccess) {
            ctx->stream_hi = nullptr;
            cudaGetLastError();
        }
    }
    ctx->pinned_cap = 1 << 16;
    if (cudaHostAlloc(&ctx->pinned, ctx->pinned_cap, cudaHostAllocDefault) != cudaSuccess) {
        cudaStreamDestroy(ctx->stream);
        delete ctx;
        return B2N_ERR_CUDA;
    }
    *out = ctx;
    return B2N_OK;
}

void b2n_free(b2n_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    DevBuf* bufs[] = {&ctx->b_ctrs, &ctx->b_ams, &ctx->b_axesT, &ctx->b_logvols, &ctx->in0, &ctx->in1,
                      &ctx->in2, &ctx->in3, &ctx->out0, &ctx->out1, &ctx->out2, &ctx->out3,
                      &ctx->out4, &ctx->out5, &ctx->out6, &ctx->out7, &ctx->scratch0,
                      &ctx->scratch1, &ctx->scratch2, &ctx->scratch3, &ctx->scratch4,
                      &ctx->scratch5, &ctx->work0, &ctx->work1, &ctx->wl_order, &ctx->wl_cta, &ctx->spec};
    if (ctx->stream_side) cudaStreamSynchronize(ctx->stream_side);
    if (ctx->stream_side2) cudaStreamSynchronize(ctx->stream_side2);
    for (DevBuf* b : bufs) b->release();
    b2n_peer_release(ctx);
    b2n_ns_release(ctx);
    b2n_friends_release(ctx);
    for (void* p : ctx->model_allocs) cudaFree(p);
    if (ctx->ev0) { cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1); }
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->stream_hi) cudaStreamDestroy(ctx->stream_hi);
    if (ctx->ev_block) cudaEventDestroy(ctx->ev_block);
    if (ctx->stream_side) cudaStreamDestroy(ctx->stream_side);
    if (ctx->ev_side) cudaEventDestroy(ctx->ev_side);
    if (ctx->ev_side_go) cudaEventDestroy(ctx->ev_side_go);
    if (ctx->stream_side2) cudaStreamDestroy(ctx->stream_side2);
    if (ctx->ev_side2) cudaEventDestroy(ctx->ev_side2);
    if (ctx->ev_side2_go) cudaEventDestroy(ctx->ev_side2_go);
    delete ctx;
}

int b2n_set_stream(b2n_ctx* ctx, void* s) {
    if (!ctx) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (s == nullptr) {
        B2N_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    } else {
        ctx->stream = (cudaStream_t)s;
        ctx->own_stream = false;
    }
    return B2N_OK;
}

int b2n_set_pointer_mode(b2n_ctx* ctx, int mode) {
    if (!ctx || (mode != B2N_PTR_HOST && mode != B2N_PTR_DEVICE)) return B2N_ERR_ARG;
    ctx->ptr_mode = mode;
    return B2N_OK;
}

}  // extern "C"
__global__ void b2n_noop_kernel(int* p) { if (p && threadIdx.x == 9999) *p = 0; }
extern "C" {

int b2n_debug_launch_rate(b2n_ctx* ctx, int32_t nlaunch, double* us_per_launch) {
    if (!ctx || nlaunch < 1 || !us_per_launch) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    for (int i = 0; i < nlaunch; i++) b2n_noop_kernel<<<1, 32, 0, ctx->stream>>>(nullptr);
    clock_gettime(CLOCK_MONOTONIC, &t1);                     // host time to ENQUEUE (the queue may back-pressure)
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    B2N_CUDA(ctx, cudaGetLastError());
    ctx->launches += nlaunch;
    *us_per_launch = ((t1.tv_sec - t0.tv_sec) * 1e6 + (t1.tv_nsec - t0.tv_nsec) * 1e-3) / nlaunch;
    return B2N_OK;
}

int b2n_set_start_rows(b2n_ctx* ctx, const int32_t* idx, int64_t nrows) {
    if (!ctx || (idx && nrows < 1)) return B2N_ERR_ARG;
    ctx->start_idx = idx;
    ctx->start_nrows = idx ? nrows : 0;
    return B2N_OK;
}

int b2n_set_chain_pack(b2n_ctx* ctx, int32_t chains_per_cta) {
    if (!ctx || chains_per_cta < 1) return B2N_ERR_ARG;
    ctx->min_cpc = chains_per_cta;
    return B2N_OK;
}

int b2n_synchronize(b2n_ctx* ctx) {
    if (!ctx) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B2N_OK;
}

int64_t b2n_launch_count(b2n_ctx* ctx) { return ctx ? ctx->launches : 0; }

int b2n_set_timing(b2n_ctx* ctx, int enabled) {
    if (!ctx) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    if (enabled && !ctx->ev0) {
        B2N_CUDA(ctx, cudaEventCreate(&ctx->ev0));
        B2N_CUDA(ctx, cudaEventCreate(&ctx->ev1));
    }
    ctx->timing = enabled ? 1 : 0;
    ctx->ev_valid = false;
    return B2N_OK;
}

double b2n_last_kernel_ms(b2n_ctx* ctx) {
    if (!ctx || !ctx->ev_valid) return -1.0;
    if (cudaEventSynchronize(ctx->ev1) != cudaSuccess) return -1.0;
    float ms = -1.f;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) != cudaSuccess) return -1.0;
    return (double)ms;
}

static int upload(b2n_ctx* ctx, const double* h, size_t count, const double** d) {
    *d = nullptr;
    if (!h || count == 0) return B2N_OK;
    void* p = nullptr;
    B2N_CUDA(ctx, cudaMalloc(&p, count * sizeof(double)));
    ctx->model_allocs.push_back(p);
    B2N_CUDA(ctx, cudaMemcpy(p, h, count * sizeof(double), cudaMemcpyHostToDevice));
    *d = (const double*)p;
    return B2N_OK;
}

int b2n_model_create(b2n_ctx* ctx, const b2n_model_desc* d, int32_t* id) {
    if (!ctx || !d || !id || d->ndim < 1) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = d->ndim;
    B2nModel m;
    memset(&m, 0, sizeof(m));
    m.ndim = d->ndim;
    m.prior_kind = d->prior_kind;
    m.like_kind = d->like_kind;
    m.s0 = d->like_s0; m.s1 = d->like_s1; m.s2 = d->like_s2;
    if (d->prior_kind < 0 || d->prior_kind > B2N_PRIOR_NORMAL_PPF) return B2N_ERR_ARG;
    if (d->like_kind < 0 || d->like_kind > B2N_LIKE_REGION2D) return B2N_ERR_ARG;
    if (d->like_kind == B2N_LIKE_REGION2D && d->ndim < 2) return B2N_ERR_ARG;
    if (d->prior_kind != B2N_PRIOR_IDENTITY && (!d->prior_p0 || !d->prior_p1)) return B2N_ERR_ARG;
    if (d->like_kind != B2N_LIKE_EGGBOX && d->like_kind != B2N_LIKE_REGION2D && !d->like_vec0) return B2N_ERR_ARG;
    if ((d->like_kind == B2N_LIKE_GAUSS_DIAG || d->like_kind == B2N_LIKE_SHELLS) && !d->like_vec1)
        return B2N_ERR_ARG;
    if (d->like_kind == B2N_LIKE_GAUSS_PREC && !d->like_mat) return B2N_ERR_ARG;
    B2N_TRY(upload(ctx, d->prior_p0, n, &m.pp0));
    B2N_TRY(upload(ctx, d->prior_p1, n, &m.pp1));
    B2N_TRY(upload(ctx, d->like_vec0, n, &m.lv0));
    B2N_TRY(upload(ctx, d->like_vec1, n, &m.lv1));
    B2N_TRY(upload(ctx, d->like_mat, n * n, &m.lmat));
    ctx->models.push_back(m);
    *id = (int32_t)ctx->models.size() - 1;
    return B2N_OK;
}

int b2n_bound_set(b2n_ctx* ctx, int32_t K, int32_t nc, const double* ctrs, const double* ams,
                  const double* axes, const double* logvols) {
    if (!ctx || K < 1 || nc < 1 || !axes) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t mat = (size_t)nc * nc;
    // axes are stored TRANSPOSED on the device (axesT[k][j*nc+i] = axes[k][i][j]) so
    // that a warp computing rows i = lane, lane+32, .. of axes @ x reads consecutive
    // addresses for a fixed column j.
    std::vector<double> t(mat * K);
    for (int k = 0; k < K; k++)
        for (int i = 0; i < nc; i++)
            for (int j = 0; j < nc; j++) t[k * mat + (size_t)j * nc + i] = axes[k * mat + (size_t)i * nc + j];
    // the previous bound may still be in use by enqueued kernels
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    B2N_CUDA(ctx, ctx->b_axesT.ensure(mat * K * sizeof(double)));
    B2N_CUDA(ctx, cudaMemcpy(ctx->b_axesT.p, t.data(), mat * K * sizeof(double), cudaMemcpyHostToDevice));
    if (ctrs && ams && logvols) {
        B2N_CUDA(ctx, ctx->b_ctrs.ensure((size_t)K * nc * sizeof(double)));
        B2N_CUDA(ctx, ctx->b_ams.ensure(mat * K * sizeof(double)));
        B2N_CUDA(ctx, ctx->b_logvols.ensure((size_t)K * sizeof(double)));
        B2N_CUDA(ctx, cudaMemcpy(ctx->b_ctrs.p, ctrs, (size_t)K * nc * sizeof(double), cudaMemcpyHostToDevice));
        B2N_CUDA(ctx, cudaMemcpy(ctx->b_ams.p, ams, mat * K * sizeof(double), cudaMemcpyHostToDevice));
        B2N_CUDA(ctx, cudaMemcpy(ctx->b_logvols.p, logvols, (size_t)K * sizeof(double), cudaMemcpyHostToDevice));
        ctx->h_logvols.assign(logvols, logvols + K);
    } else {
        ctx->h_logvols.clear();
    }
    ctx->bK = K;
    ctx->bn = nc;
    ctx->bound_serial++;
    return B2N_OK;
}

}  // extern "C"

// axes (K x nc x nc, row-major) -> axesT[k][j*nc+i] = axes[k][i][j], on the device
__global__ void transpose_axes_kernel(const double* __restrict__ axes, double* __restrict__ axesT, int K, int nc) {
    const size_t mat = (size_t)nc * nc, tot = mat * K;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (size_t)gridDim.x * blockDim.x) {
        const size_t k = e / mat, r = e - k * mat;
        const int j = (int)(r / nc), i = (int)(r - (size_t)j * nc);
        axesT[e] = axes[k * mat + (size_t)i * nc + j];
    }
}

// b2n_bound_set for arrays that already live on the device (b2n_ns_update_bound): no host staging.
// logvols: HOST copy (K), needed for the volume-weighted ellipsoid pick of the uniform sampler.
int b2n_bound_set_dev(b2n_ctx* ctx, int K, int nc, const double* dctrs, const double* dams, const double* daxes,
                      const double* h_logvols) {
    const size_t mat = (size_t)nc * nc;
    B2N_CUDA(ctx, ctx->b_axesT.ensure(mat * K * sizeof(double)));
    B2N_CUDA(ctx, ctx->b_ctrs.ensure((size_t)K * nc * sizeof(double)));
    B2N_CUDA(ctx, ctx->b_ams.ensure(mat * K * sizeof(double)));
    B2N_CUDA(ctx, ctx->b_logvols.ensure((size_t)K * sizeof(double)));
    cudaStream_t st = ctx->stream;       // stream order: kernels enqueued before still see the previous bound
    transpose_axes_kernel<<<(unsigned)std::min<size_t>((mat * K + 255) / 256, 1024), 256, 0, st>>>(daxes, ctx->b_axesT.as<double>(), K, nc);
    B2N_LAUNCH_CHECK(ctx);
    B2N_CUDA(ctx, cudaMemcpyAsync(ctx->b_ctrs.p, dctrs, (size_t)K * nc * sizeof(double), cudaMemcpyDeviceToDevice, st));
    B2N_CUDA(ctx, cudaMemcpyAsync(ctx->b_ams.p, dams, mat * K * sizeof(double), cudaMemcpyDeviceToDevice, st));
    ctx->h_logvols.assign(h_logvols, h_logvols + K);
    B2N_CUDA(ctx, cudaMemcpyAsync(ctx->b_logvols.p, ctx->h_logvols.data(), (size_t)K * sizeof(double), cudaMemcpyHostToDevice, st));
    ctx->bK = K;
    ctx->bn = nc;
    ctx->bound_serial++;
    return B2N_OK;
}

extern "C" {


}  // extern "C"

// ---- batched model evaluation: one warp per point -------------------------------------
template <int LIKE>
__global__ void __launch_bounds__(256) model_eval_kernel(B2nModel m, const double* __restrict__ u,
                                                         int64_t M, double* __restrict__ v,
                                                         double* __restrict__ logl) {
    extern __shared__ double sm[];
    const int n = m.ndim;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    double* vv = sm + (size_t)warp * 2 * n;
    double* work = vv + n;
    for (int64_t p = (int64_t)blockIdx.x * wpb + warp; p < M; p += (int64_t)gridDim.x * wpb) {
        for (int i = lane; i < n; i += 32) {
            const double x = prior_1d(m, i, u[p * n + i]);
            vv[i] = x;
            if (v) v[p * n + i] = x;
        }
        __syncwarp();
        const double l = warp_loglike<LIKE>(m, m.lmat, vv, work, lane);
        if (lane == 0) logl[p] = l;
        __syncwarp();
    }
}

extern "C" int b2n_model_eval(b2n_ctx* ctx, int32_t id, const double* u, int64_t M, double* v,
                              double* logl) {
    if (!ctx || id < 0 || id >= (int)ctx->models.size() || !u || !logl || M < 0) return B2N_ERR_ARG;
    if (M == 0) return B2N_OK;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    const B2nModel m = ctx->models[id];
    const size_t n = m.ndim;
    const void *du;
    void *dv, *dl;
    B2N_TRY(b2n_in(ctx, ctx->in0, u, M * n * sizeof(double), &du));
    B2N_TRY(b2n_out(ctx, ctx->out0, v, M * n * sizeof(double), &dv));
    B2N_TRY(b2n_out(ctx, ctx->out1, logl, M * sizeof(double), &dl));
    const int threads = 256, wpb = threads / 32;
    const size_t smem = (size_t)wpb * 2 * n * sizeof(double);
    int64_t blocks = (M + wpb - 1) / wpb;
    if (blocks > (int64_t)ctx->sm_count * 8) blocks = (int64_t)ctx->sm_count * 8;
#define CALL(L)                                                                                   \
    if (smem > 48 * 1024)                                                                          \
        B2N_TRY(b2n_func_smem(ctx, (const void*)(model_eval_kernel<L>), (size_t)(smem))); \
    model_eval_kernel<L><<<(unsigned)blocks, threads, smem, ctx->stream>>>(                         \
        m, (const double*)du, M, (double*)dv, (double*)dl);
    B2N_DISPATCH_LIKE(m.like_kind, CALL)
#undef CALL
    B2N_LAUNCH_CHECK(ctx);
    B2N_TRY(b2n_out_done(ctx, v, dv, M * n * sizeof(double)));
    B2N_TRY(b2n_out_done(ctx, logl, dl, M * sizeof(double)));
    return b2n_finish(ctx);
}
