// b2n_common.cuh -- context, scratch memory and small device helpers shared by
// all translation units of libb200nest.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "../../include/b200nest.h"

#define B2N_WARP 32
#define B2N_FULL 0xffffffffu

// ---- device-side model descriptor (passed by value to kernels) -------------
struct B2nModel {
    int ndim, prior_kind, like_kind, pad;
    const double* pp0;   // device
    const double* pp1;
    const double* lv0;
    const double* lv1;
    const double* lmat;
    double s0, s1, s2;
};

// growable device buffer
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() { return reinterpret_cast<T*>(p); }
};

// ---- peer exchange (multi-GPU gather fused into the chain kernels, b2n_peer.cu) ----------
// Window layout: 256-byte header { u64 arrive @0 | u32 err @8 | u32 done @64 } then two slots
// (call parity) of { u (R x n f64) | v (R x n f64) | logl (R f64) | 4 x (R i32) }, R = total rows,
// every array 256-byte aligned.  The same (R, n) gives the same layout on every rank.
#define B2N_PEER_HDR 256
struct PeerSet {               // passed by value to the chain kernels; world == 0: exchange off
    int world = 0, rank = 0;
    char* base[B2N_MAX_PEERS] = {nullptr};
    unsigned long long target = 0;     // own arrive counter once every rank has arrived
};
struct PeerState {
    int world = 0, rank = 0;
    char* win = nullptr;               // own window
    size_t win_bytes = 0;
    char* base[B2N_MAX_PEERS] = {nullptr};
    bool opened[B2N_MAX_PEERS] = {false};      // mapped through cudaIpcOpenMemHandle
    int64_t row0 = 0, total = 0;       // gather mode when total > 0
    uint64_t epoch = 0;                // gather-mode calls so far (same on all ranks)
    uint64_t off[7] = {0};             // byte offsets of the arrays of the last call
    unsigned int* err_host = nullptr;  // pinned mailbox for the window's err word
};

// ---- device-paced launches (b2n_ns.cu): the per-round arguments of a chain kernel live in HBM,
// written by the previous kernel on the stream, so that consecutive nested-sampling rounds need
// no host round trip.  A chain kernel given a B2nDyn reads its threshold / scale / chain ids /
// CTA count from it and returns at once when `skip` is set.
struct B2nDyn {
    double loglstar, scale;
    unsigned long long chain0;
    int skip, ncta, doubling, pad;
};
struct DynLaunch {
    bool active = false;         // the next chain entry call is device-paced
    bool plan_only = false;      // ... and only reports chains_per_cta (no launch)
    const B2nDyn* dev = nullptr;
    const int* order = nullptr;  // device worklist (same layout as b2n_build_worklist's)
    const int3* cta = nullptr;
    int max_cta = 0;             // grid size: upper bound of the CTA count
    int cpc = 0;                 // out: chains per CTA the entry point planned for
};

struct b2n_ns;                   // device-resident nested-sampling run (b2n_ns.cu)

struct b2n_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream_hi = nullptr;   // highest-priority twin of the own stream: bound updates of a device-resident run
    bool own_stream = true;
    int ptr_mode = B2N_PTR_HOST;
    int sm_count = 148;
    int max_smem_optin = 0;
    int64_t launches = 0;
    int timing = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t ev_block = nullptr;     // blocking-sync event: long waits of a context that shares the GPU sleep, not spin
    bool ev_valid = false;
    char err[512] = {0};
    std::vector<B2nModel> models;
    std::vector<void*> model_allocs;
    // resident bound
    int bK = 0, bn = 0;
    DevBuf b_ctrs, b_ams, b_axesT, b_logvols;
    unsigned long long bound_serial = 0;   // bumped by every b2n_bound_set / b2n_bound_set_dev (who holds the bound)
    std::vector<double> h_logvols;
    // staging (host-pointer mode) and scratch
    DevBuf in0, in1, in2, in3, out0, out1, out2, out3, out4, out5, out6, out7;
    DevBuf scratch0, scratch1, scratch2, scratch3, scratch4, scratch5;
    DevBuf work0, work1;
    void* pinned = nullptr;     // small pinned host mailbox
    size_t pinned_cap = 0;
    PeerState peer;
    DynLaunch dyn;
    b2n_ns* ns = nullptr;
    void* friends = nullptr;    // resident RadFriends / SupFriends bound (b2n_friends.cu)
    const int32_t* start_idx = nullptr;   // b2n_set_start_rows: the NEXT rwalk call reads its start points as rows of u0
    int64_t start_nrows = 0;
    int min_cpc = 1;            // b2n_set_chain_pack: at least this many chains per CTA (see include/b200nest.h)
    int bound_fast_skip = 0;    // b2n_multi_decompose: updates left to skip the Cholesky candidate path
    // speculative eigen fit of the root node, concurrent with the candidate tree (b2n_bounding.cu: b2n_spec_root_*)
    cudaStream_t stream_side = nullptr, stream_side2 = nullptr;   // side2: the major-axis half of the candidate fits
    cudaEvent_t ev_side = nullptr, ev_side_go = nullptr, ev_side2 = nullptr, ev_side2_go = nullptr;
    DevBuf spec;
    bool zc_enabled = false;    // chain entry points, host-pointer mode: pinned caller buffers are used in place
    // cached chain worklist of the single-ellipsoid case (identity order, equal CTAs): rebuilt only when
    // (Q, chains per CTA) change -- saves two small pageable H2D copies per queue fill
    DevBuf wl_order, wl_cta;
    int64_t wl_Q = -1;
    int wl_cpc = 0, wl_ncta = 0;
};
// cudaFuncAttributeMaxDynamicSharedMemorySize, raised ONCE per (device, kernel) and never lowered: the attribute is
// process-wide per device, so two contexts of different problem sizes must not shrink each other's limit, and a driver
// call per launch is a lock every replica thread would queue on (b2n_ctx.cu)
int b2n_func_smem(b2n_ctx* ctx, const void* func, size_t bytes);
void b2n_ns_release(b2n_ctx* ctx);
void b2n_friends_release(b2n_ctx* ctx);
int b2n_bound_set_dev(b2n_ctx* ctx, int K, int nc, const double* dctrs, const double* dams, const double* daxes,
                      const double* h_logvols);
// friends mode of the device-resident rounds (b2n_friends.cu, used by b2n_ns.cu; all pointers device arrays):
//   y = x @ T for N rows (friends_transform_kernel); cov *= f^2, am /= f^2, axes *= f, axes_inv /= f (the host class's
//   scale_to_logvol arithmetic); UniformBoundSampler.sample with the centres `ctrs` (N rows), device-paced (ctx->dyn)
int b2n_friends_transform_dev(b2n_ctx* ctx, const double* x, int N, int n, const double* T, double* y);
int b2n_friends_rescale_dev(b2n_ctx* ctx, int n, double* cov, double* am, double* axes, double* axes_inv, double f);
int b2n_friends_unif_dev(b2n_ctx* ctx, const b2n_chain_args* a, int N, int kind, const double* ctrs, const double* ctrs_t,
                         const double* axes, const double* axes_inv, double* u, double* v, double* logl, int32_t* ncall,
                         int32_t* nprop, uint32_t* flags);

// gather-mode plumbing shared by the chain entry points (b2n_peer.cu).  b2n_peer_begin: when
// gather mode is on, point the 7 output arrays at this rank's rows of its own window and fill
// `ps`; returns through *on whether it did.  b2n_peer_end: copy the gathered arrays (total rows)
// to the caller's pointers and fetch the error word; b2n_peer_finish replaces b2n_finish.
int b2n_peer_begin(b2n_ctx* ctx, int n, PeerSet* ps, void** dev7, bool* on);
int b2n_peer_end(b2n_ctx* ctx, int n, void* const* user7);
int b2n_peer_finish(b2n_ctx* ctx, bool on);
void b2n_peer_release(b2n_ctx* ctx);

#define B2N_CUDA(ctx, call)                                                        \
    do {                                                                           \
        cudaError_t e_ = (call);                                                   \
        if (e_ != cudaSuccess) {                                                   \
            snprintf((ctx)->err, sizeof((ctx)->err), "%s:%d %s: %s", __FILE__,     \
                     __LINE__, #call, cudaGetErrorString(e_));                     \
            return B2N_ERR_CUDA;                                                   \
        }                                                                          \
    } while (0)

#define B2N_TRY(call)                         \
    do {                                      \
        int s_ = (call);                      \
        if (s_ != B2N_OK) return s_;          \
    } while (0)

#define B2N_TIME_BEGIN(ctx) do { if ((ctx)->timing) cudaEventRecord((ctx)->ev0, (ctx)->stream); } while (0)
#define B2N_TIME_END(ctx) do { if ((ctx)->timing) { cudaEventRecord((ctx)->ev1, (ctx)->stream); (ctx)->ev_valid = true; } } while (0)

#define B2N_LAUNCH_CHECK(ctx)                 \
    do {                                      \
        (ctx)->launches++;                    \
        B2N_CUDA(ctx, cudaGetLastError());    \
    } while (0)

// Blocking copy ON THE CONTEXT'S STREAM (cudaMemcpy proper runs on the legacy default stream, a process-wide object
// every replica thread would serialise on).
static inline cudaError_t b2n_copy_sync(b2n_ctx* ctx, void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) {
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind, ctx->stream);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(ctx->stream);
}

static inline int b2n_fail(b2n_ctx* ctx, int status, const char* msg) {
    snprintf(ctx->err, sizeof(ctx->err), "%s", msg);
    return status;
}

// Zero-copy for PINNED caller buffers (host-pointer mode, chain entry points only: their inputs are read
// once and their outputs written once).  Under UVA a cudaHostAlloc'ed buffer is addressable from the device
// by its host address: the kernel then reads the start points / writes the finished chains straight over
// PCIe -- the transfer overlaps the kernel instead of following it as a DMA copy.  Pageable memory (plain
// numpy arrays) keeps the staged path.
static inline bool b2n_zc_ok(b2n_ctx* ctx, const void* p) {
    if (!ctx->zc_enabled || p == nullptr) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost && a.devicePointer == p;
}
struct ZcScope {          // enables zero-copy for the lifetime of a chain entry call
    b2n_ctx* c;
    explicit ZcScope(b2n_ctx* ctx) : c(ctx) {
        const char* e = getenv("B2N_ZERO_COPY");
        c->zc_enabled = c->ptr_mode == B2N_PTR_HOST && !(e && e[0] == '0');
    }
    ~ZcScope() { c->zc_enabled = false; }
};

// Input staging: returns a device pointer for `src` (copying when in host mode).
static inline int b2n_in(b2n_ctx* ctx, DevBuf& buf, const void* src, size_t bytes,
                         const void** dev) {
    if (ctx->ptr_mode == B2N_PTR_DEVICE || src == nullptr || bytes == 0 || b2n_zc_ok(ctx, src)) {
        *dev = src;
        return B2N_OK;
    }
    B2N_CUDA(ctx, buf.ensure(bytes));
    B2N_CUDA(ctx, cudaMemcpyAsync(buf.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    *dev = buf.p;
    return B2N_OK;
}
// Host-resident argument that is needed on the device in both modes.
static inline int b2n_in_host(b2n_ctx* ctx, DevBuf& buf, const void* src, size_t bytes,
                              const void** dev) {
    if (src == nullptr || bytes == 0) { *dev = nullptr; return B2N_OK; }
    B2N_CUDA(ctx, buf.ensure(bytes));
    B2N_CUDA(ctx, cudaMemcpyAsync(buf.p, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    *dev = buf.p;
    return B2N_OK;
}
// Output staging: device pointer to write into.
static inline int b2n_out(b2n_ctx* ctx, DevBuf& buf, void* dst, size_t bytes, void** dev) {
    if (dst == nullptr) { *dev = nullptr; return B2N_OK; }
    if (ctx->ptr_mode == B2N_PTR_DEVICE || b2n_zc_ok(ctx, dst)) { *dev = dst; return B2N_OK; }
    B2N_CUDA(ctx, buf.ensure(bytes));
    *dev = buf.p;
    return B2N_OK;
}
static inline int b2n_out_done(b2n_ctx* ctx, void* dst, const void* dev, size_t bytes) {
    if (dst == nullptr || ctx->ptr_mode == B2N_PTR_DEVICE || dev == dst) return B2N_OK;   // dev == dst: written in place
    B2N_CUDA(ctx, cudaMemcpyAsync(dst, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return B2N_OK;
}
static inline int b2n_finish(b2n_ctx* ctx) {
    if (ctx->ptr_mode == B2N_PTR_HOST) B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B2N_OK;
}

// ---- warp helpers ----------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(B2N_FULL, v, o);
    return v;
}
__device__ __forceinline__ double warp_prod(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v *= __shfl_xor_sync(B2N_FULL, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(B2N_FULL, v, o));
    return v;
}
__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(B2N_FULL, v, o));
    return v;
}

// y_i = sum_j M[j*ld + i] * x[j] for the two rows i0 = base+lane, i1 = i0+32
// (column-major panel: lanes read consecutive addresses; x is a warp broadcast).
// Four accumulators per row keep the FP64 pipe busy despite the DFMA latency.
__device__ __forceinline__ void warp_matvec2(const double* __restrict__ M, int ld, int ncols,
                                             const double* __restrict__ x, int i0, int nrows,
                                             double& y0, double& y1) {
    const int i1 = i0 + 32;
    const bool r0 = i0 < nrows, r1 = i1 < nrows;
    const int a0 = r0 ? i0 : 0, a1 = r1 ? i1 : 0;
    double p0 = 0, p1 = 0, q0 = 0, q1 = 0;
    int j = 0;
    for (; j + 1 < ncols; j += 2) {
        const double xa = x[j], xb = x[j + 1];
        p0 = fma(M[(size_t)j * ld + a0], xa, p0);
        p1 = fma(M[(size_t)j * ld + a1], xa, p1);
        q0 = fma(M[(size_t)(j + 1) * ld + a0], xb, q0);
        q1 = fma(M[(size_t)(j + 1) * ld + a1], xb, q1);
    }
    if (j < ncols) {
        const double xa = x[j];
        p0 = fma(M[(size_t)j * ld + a0], xa, p0);
        p1 = fma(M[(size_t)j * ld + a1], xa, p1);
    }
    y0 = r0 ? p0 + q0 : 0.0;
    y1 = r1 ? p1 + q1 : 0.0;
}
