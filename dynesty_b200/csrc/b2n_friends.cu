// b2n_friends.cu -- RadFriends / SupFriends: the bound made of one ball / cube per live point
// (reference bounding.py:734-996 RadFriends, :999-1263 SupFriends, radii helpers :1651-1705).  SURVEY 8(f) row 3.
//
// What the reference does per update (bounding.py:874-958 / 1142-1226):
//   1. clusters = single-linkage tree of the points under the CURRENT metric `am`, cut at Mahalanobis distance 1
//      (:966-977)  ==  connected components of the graph {(i, j): d_M(i, j) <= 1};
//      covariance of the points re-centred on their cluster means (:979-993), np.cov (ddof = 1);
//   2. am = pinvh(cov), axes = sqrtm(cov), axes_inv = pinvh(axes) (:923-925)  -- all from ONE symmetric
//      eigen-decomposition of cov;
//   3. points_t = points @ axes_inv; radius = max over points of the distance to the nearest OTHER point
//      (leave-one-out, :1683-1705; Euclidean for balls, Chebyshev for cubes), or -- bootstrap -- the max over
//      resamples of the largest out-of-bag -> nearest in-bag distance (:1651-1680);
//   4. cov *= r^2, am /= r^2, axes *= r, axes_inv /= r; logvol = prefactor - slogdet(am) / 2.
// Queries: within / overlap / contains = count of centres with |(c_i - x) @ axes_inv| <= 1 (:776-795, 1042-1062);
// sample = random centre + random offset in the ball / cube, accepted with probability 1/q (:797-831, 1065-1100).
//
// B200 mapping.  All of it is brute force over pairs -- which is also what the reference does for the queries,
// and what its KD-trees approximate for the radii -- and brute force over N^2 n with N ~ 10^3 is a few 10^8 flop:
//   friends_transform_kernel   y = x @ T (T = metric square root), one warp per point
//   friends_adj_kernel         adjacency bit matrix of {|y_i - y_j|^2 <= 1}: one thread per (row, 32-column word)
//   friends_label_kernel       min-label propagation over the bit matrix + pointer jumping, to the fixed point
//   friends_center_kernel      per-cluster mean (fixed-order reduction, one CTA per cluster) and re-centring
//   (moments: the node kernels of b2n_bounding.cu on the re-centred block as ONE node: np.cov, ddof = 1)
//   friends_metric_kernel      one CTA: Jacobi eigen-decomposition (b2n_jacobi.cuh) -> am, axes, axes_inv, ln det
//   friends_nn_kernel          nearest-neighbour distance of every point to a masked subset (LOO / bootstrap)
//   friends_overlap_kernel     q for a batch of query points, one warp per query
//   friends_unif_kernel        UniformBoundSampler.sample with this bound: one warp per chain
// Everything is deterministic (no atomics on floating point, fixed reduction orders).
#include "b2n_jacobi.cuh"
#include "b2n_bounding.cuh"
#include <algorithm>
#include <math_constants.h>
#include <vector>

#define B2N_UNIF_MAX_DRAWS 20000000

struct FriendsState {
    int kind = 0, N = 0, n = 0;       // kind 0 balls, 1 cubes
    DevBuf ctrs, ctrs_t, axes, axes_inv;
};

static FriendsState* friends_of(b2n_ctx* ctx) {
    if (!ctx->friends) ctx->friends = new FriendsState();
    return reinterpret_cast<FriendsState*>(ctx->friends);
}

void b2n_friends_release(b2n_ctx* ctx) {
    if (!ctx || !ctx->friends) return;
    FriendsState* f = reinterpret_cast<FriendsState*>(ctx->friends);
    f->ctrs.release(); f->ctrs_t.release(); f->axes.release(); f->axes_inv.release();
    delete f;
    ctx->friends = nullptr;
}

// y[i][j] = sum_k x[i][k] T[k][j]   (row vector times matrix), one warp per point
__global__ void __launch_bounds__(256) friends_transform_kernel(const double* __restrict__ x, int N, int n,
                                                                const double* __restrict__ T, double* __restrict__ y) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= N) return;
    const double* xi = x + (size_t)warp * n;
    for (int j = lane; j < n; j += 32) {
        double s = 0.0;
        for (int k = 0; k < n; k++) s = fma(xi[k], __ldg(T + (size_t)k * n + j), s);
        y[(size_t)warp * n + j] = s;
    }
}

// bit (i, j) of adj = |y_i - y_j| <= 1 (Euclidean); one thread per (row i, word w), summation in index order
__global__ void __launch_bounds__(256) friends_adj_kernel(const double* __restrict__ y, int N, int n, int W,
                                                          uint32_t* __restrict__ adj) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)N * W) return;
    const int i = (int)(t / W), w = (int)(t - (size_t)i * W);
    const double* yi = y + (size_t)i * n;
    uint32_t bits = 0;
    for (int b = 0; b < 32; b++) {
        const int j = w * 32 + b;
        if (j >= N) break;
        const double* yj = y + (size_t)j * n;
        double s = 0.0;
        for (int k = 0; k < n; k++) { const double d = yi[k] - yj[k]; s = fma(d, d, s); }
        if (sqrt(s) <= 1.0) bits |= (1u << b);
    }
    adj[t] = bits;
}

// one sweep: lab_out[i] = min(lab_in[i], min_{j adjacent} lab_in[j]), then one pointer jump; *changed |= any change
__global__ void __launch_bounds__(256) friends_label_kernel(const uint32_t* __restrict__ adj, int N, int W,
                                                            const int* __restrict__ lin, int* __restrict__ lout,
                                                            int* __restrict__ changed) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= N) return;
    int m = lin[warp];
    for (int w = lane; w < W; w += 32) {
        uint32_t bits = adj[(size_t)warp * W + w];
        while (bits) {
            const int b = __ffs(bits) - 1;
            bits &= bits - 1;
            m = min(m, lin[w * 32 + b]);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(B2N_FULL, m, o));
    m = min(m, lin[m]);                          // pointer jump (labels only decrease: reading lin is safe)
    if (lane == 0) {
        lout[warp] = m;
        if (m != lin[warp]) *changed = 1;
    }
}

// one CTA per cluster: mean of its rows (segment [start, start+count) of perm), over[pos] = x[row] - mean
__global__ void __launch_bounds__(256) friends_center_kernel(const double* __restrict__ x, int n, const int* __restrict__ perm,
                                                             const int2* __restrict__ seg, double* __restrict__ over) {
    extern __shared__ double fsm[];
    const int start = seg[blockIdx.x].x, count = seg[blockIdx.x].y;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        double s = 0.0;
        for (int r = 0; r < count; r++) s += x[(size_t)perm[start + r] * n + j];      // index order: np.mean's pairwise
        fsm[j] = s / (double)count;                                                    // sum differs by O(eps) only
    }
    __syncthreads();
    for (int e = threadIdx.x; e < count * n; e += blockDim.x) {
        const int r = e / n, j = e - r * n;
        over[(size_t)(start + r) * n + j] = x[(size_t)perm[start + r] * n + j] - fsm[j];
    }
}

// One CTA: cov -> eigen -> am = pinvh(cov), axes = sqrtm(cov), axes_inv = pinvh(axes), ln det(am).
// out: [am | axes | axes_inv] (n*n each), scal[0] = ln det(am) (-inf if an eigenvalue was cut), scal[1] = #cut
__global__ void __launch_bounds__(1024) friends_metric_kernel(const double* __restrict__ cov, int n, int ld,
                                                              double* __restrict__ out, double* __restrict__ scal) {
    extern __shared__ double fsm[];
    const int tid = threadIdx.x, T = blockDim.x;
    const int half = ((n + 1) & ~1) >> 1;
    double* cc = fsm;
    double* ss = cc + half;
    double* lam = ss + half;
    double* ia = lam + n;        // 1/lambda (pinvh(cov))
    double* sq = ia + n;         // sqrt(lambda)
    double* isq = sq + n;        // 1/sqrt(lambda) (pinvh(axes))
    double* red = isq + n;
    double* A = red + 32;
    double* VT = A + (size_t)n * ld;
    for (int e = tid; e < n * n; e += T) {
        const int i = e / n, j = e - i * n;
        A[(size_t)i * ld + j] = 0.5 * (cov[(size_t)i * n + j] + cov[(size_t)j * n + i]);
        VT[(size_t)i * ld + j] = (i == j) ? 1.0 : 0.0;
    }
    __syncthreads();
    jacobi_eig(A, VT, n, ld, cc, ss, red);
    for (int k = tid; k < n; k += T) lam[k] = A[(size_t)k * ld + k];
    __syncthreads();
    if (tid == 0) {
        double mx = 0.0;
        for (int k = 0; k < n; k++) mx = fmax(mx, fabs(lam[k]));
        const double eps = 2.220446049250313e-16;
        const double cut = (double)n * eps * mx;                       // scipy.linalg.pinvh: max(M, N) eps max|lambda|
        double smx = 0.0;
        for (int k = 0; k < n; k++) { sq[k] = sqrt(fmax(lam[k], 0.0)); smx = fmax(smx, sq[k]); }
        const double cut2 = (double)n * eps * smx;
        double ld_am = 0.0;
        int ncut = 0;
        for (int k = 0; k < n; k++) {
            if (fabs(lam[k]) > cut) { ia[k] = 1.0 / lam[k]; ld_am -= log(fabs(lam[k])); }
            else { ia[k] = 0.0; ncut++; }
            isq[k] = (sq[k] > cut2) ? 1.0 / sq[k] : 0.0;
        }
        scal[0] = ncut ? -CUDART_INF : ld_am;
        scal[1] = (double)ncut;
    }
    __syncthreads();
    const size_t nn = (size_t)n * n;
    for (int e = tid; e < n * n; e += T) {
        const int i = e / n, j = e - i * n;
        double a = 0.0, x = 0.0, xi = 0.0;
        for (int k = 0; k < n; k++) {
            const double vv = VT[(size_t)k * ld + i] * VT[(size_t)k * ld + j];
            a = fma(vv, ia[k], a);
            x = fma(vv, sq[k], x);
            xi = fma(vv, isq[k], xi);
        }
        out[e] = a;
        out[nn + e] = x;
        out[2 * nn + e] = xi;
    }
}

// dist[i] = min over j with mask[j] != 0 (and j != i) of |y_i - y_j|  (kind 0: Euclidean, 1: Chebyshev);
// rows with want[i] == 0 are skipped (dist = -1).  One warp per row i, lanes over j, fixed-order min.
__global__ void __launch_bounds__(256) friends_nn_kernel(const double* __restrict__ y, int N, int n, int kind,
                                                         const unsigned char* __restrict__ mask,
                                                         const unsigned char* __restrict__ want, double* __restrict__ dist) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= N) return;
    if (want && !want[warp]) { if (lane == 0) dist[warp] = -1.0; return; }
    const double* yi = y + (size_t)warp * n;
    double best = CUDART_INF;
    for (int j = lane; j < N; j += 32) {
        if (j == warp || (mask && !mask[j])) continue;
        const double* yj = y + (size_t)j * n;
        double s = 0.0;
        if (kind == 0) {
            for (int k = 0; k < n; k++) { const double d = yi[k] - yj[k]; s = fma(d, d, s); }
        } else {
            for (int k = 0; k < n; k++) s = fmax(s, fabs(yi[k] - yj[k]));
        }
        best = fmin(best, s);
    }
    best = warp_min(best);
    if (lane == 0) dist[warp] = kind == 0 ? sqrt(best) : best;
}

__global__ void friends_max_kernel(const double* __restrict__ v, int N, double* __restrict__ out) {
    __shared__ double red[32];
    double m = -CUDART_INF;
    for (int i = threadIdx.x; i < N; i += blockDim.x) m = fmax(m, v[i]);
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : -CUDART_INF;
        m = warp_max(m);
        if (threadIdx.x == 0) *out = m;
    }
}

__global__ void friends_scale_kernel(double* __restrict__ m, size_t count, double f) {
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (size_t)gridDim.x * blockDim.x) m[e] *= f;
}

// _B200Friends.scale_to_logvol (bounding.py:765-774 / 1031-1040) element by element: cov * f**2, am / f**2, axes * f,
// axes_inv / f -- the same IEEE operations as the numpy expressions (a division stays a division), so that the enlarged
// bound of the device rounds equals the host route's bit for bit
__global__ void friends_rescale_kernel(double* __restrict__ cov, double* __restrict__ am, double* __restrict__ axes,
                                       double* __restrict__ axes_inv, size_t count, double f, double f2) {
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (size_t)gridDim.x * blockDim.x) {
        cov[e] *= f2;
        am[e] /= f2;
        axes[e] *= f;
        axes_inv[e] /= f;
    }
}

// distance of the transformed query xt to centre row ct (kind 0: squared Euclidean, 1: Chebyshev)
__device__ __forceinline__ double friends_dist(const double* __restrict__ ct, const double* xt, int n, int kind) {
    double s = 0.0;
    if (kind == 0) {
        for (int k = 0; k < n; k++) { const double d = ct[k] - xt[k]; s = fma(d, d, s); }
        return sqrt(s);
    }
    for (int k = 0; k < n; k++) s = fmax(s, fabs(ct[k] - xt[k]));
    return s;
}

// q[m] = number of centres whose ball / cube contains x_m; one warp per query, x_t staged in shared memory
__global__ void __launch_bounds__(128) friends_overlap_kernel(const double* __restrict__ x, int64_t M, int n, int kind,
                                                              const double* __restrict__ ctrs_t, int N,
                                                              const double* __restrict__ axes_inv, int* __restrict__ q) {
    extern __shared__ double fsm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    double* xt = fsm + (size_t)warp * n;
    for (int64_t m = (int64_t)blockIdx.x * wpb + warp; m < M; m += (int64_t)gridDim.x * wpb) {
        const double* xm = x + m * n;
        for (int j = lane; j < n; j += 32) {
            double s = 0.0;
            for (int k = 0; k < n; k++) s = fma(xm[k], __ldg(axes_inv + (size_t)k * n + j), s);
            xt[j] = s;
        }
        __syncwarp();
        int c = 0;
        for (int i = lane; i < N; i += 32) c += friends_dist(ctrs_t + (size_t)i * n, xt, n, kind) <= 1.0 ? 1 : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(B2N_FULL, c, o);
        if (lane == 0) q[m] = c;
        __syncwarp();
    }
}

// ---- UniformBoundSampler.sample (internal_samplers.py:243-340) with a RadFriends / SupFriends bound ----------
struct FriendsUnifParams {
    B2nModel m;
    int n, N, kind, draw_only;      // draw_only: 1 = Bound.samples (no cube test / likelihood), 3 = sample(return_q)
    const double *ctrs, *ctrs_t, *axes, *axes_inv;
    const uint32_t* dimflags;
    double loglstar;
    uint64_t seed, chain0;
    int64_t Q;
    double *u, *v, *logl;
    int *ncall, *nprop;
    uint32_t* flags;
    const B2nDyn* dyn;     // device-paced launch (friends mode of b2n_ns.cu): threshold / chain ids in HBM
};

template <int LIKE>
__global__ void __launch_bounds__(128) friends_unif_kernel(const FriendsUnifParams p) {
    extern __shared__ double fsm[];
    const int n = p.n, N = p.N;
    double loglstar_ = p.loglstar;
    uint64_t chain0_ = p.chain0;
    if (p.dyn) {
        if (p.dyn->skip) return;
        loglstar_ = p.dyn->loglstar; chain0_ = p.dyn->chain0;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    double* uu = fsm + (size_t)warp * 5 * n;
    double* z = uu + n;
    double* xt = z + n;
    double* vv = xt + n;
    double* work = vv + n;
    const double inv_n = 1.0 / (double)n;
    for (int64_t q = (int64_t)blockIdx.x * wpb + warp; q < p.Q; q += (int64_t)gridDim.x * wpb) {
        ChainRng g;
        g.init(p.seed, chain0_ + (uint64_t)q);
        int ncall = 0, nprop = 0;
        uint32_t fl = 0;
        double lcur = 0.0;
        bool done = false;
        while (!done) {
            if (nprop >= B2N_UNIF_MAX_DRAWS) { fl |= 0x80000000u | B2N_WARN_UNIF_INEFFICIENT; break; }
            if (nprop == 10000) fl |= B2N_WARN_UNIF_INEFFICIENT;
            int qn = 1;
            for (;;) {                                       // bound.sample(): bounding.py:797-831 / 1065-1100
                double fac = 1.0;
                if (p.kind == 0) {                           // randsphere: normal vector, then the radius uniform
                    const double ss = rng_normals_to(g, z, n, lane);
                    const double U = rng_uniform(g);
                    fac = pow(U, inv_n) / sqrt(ss);
                } else {                                     // uniform(-1, 1, size=ndim)
                    for (int e = lane; e < n; e += 32) z[e] = 2.0 * rng_uniform_elem(g, e) - 1.0;
                    g.tick++;
                }
                __syncwarp();
                int idx = 0;
                if (N > 1) {                                 // rstate.integers(nctrs): floor(U * nctrs)
                    const double U = rng_uniform(g);
                    idx = (int)(U * (double)N);
                    idx = idx < N - 1 ? idx : N - 1;
                }
                for (int j = lane; j < n; j += 32) {         // dx = ds @ axes
                    double s = 0.0;
                    for (int k = 0; k < n; k++) s = fma(z[k], __ldg(p.axes + (size_t)k * n + j), s);
                    uu[j] = fma(fac, s, p.ctrs[(size_t)idx * n + j]);
                }
                __syncwarp();
                if (N == 1) { qn = 1; break; }
                for (int j = lane; j < n; j += 32) {
                    double s = 0.0;
                    for (int k = 0; k < n; k++) s = fma(uu[k], __ldg(p.axes_inv + (size_t)k * n + j), s);
                    xt[j] = s;
                }
                __syncwarp();
                int c = 0;
                for (int i = lane; i < N; i += 32) c += friends_dist(p.ctrs_t + (size_t)i * n, xt, n, p.kind) <= 1.0 ? 1 : 0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(B2N_FULL, c, o);
                qn = c;
                __syncwarp();
                if (qn == 1 || (p.draw_only & 2)) break;
                // (qn == 0 cannot happen mathematically -- the draw lies in the ball of centre idx -- but the two
                //  evaluation orders differ in the last bit for a point on the rim: treat it as q = 1)
                if (qn == 0) { qn = 1; break; }
                if (rng_uniform(g) < 1.0 / (double)qn) break;
            }
            nprop++;
            if (p.draw_only) {
                for (int i = lane; i < n; i += 32) vv[i] = uu[i];
                ncall = qn;
                break;
            }
            bool ok = true;
            for (int i = lane; i < n; i += 32) ok = ok && in_cube(uu[i], p.dimflags ? p.dimflags[i] : 0u);
            ok = __all_sync(B2N_FULL, ok);
            if (!ok) continue;
            for (int i = lane; i < n; i += 32) vv[i] = prior_1d(p.m, i, uu[i]);
            __syncwarp();
            lcur = warp_loglike<LIKE>(p.m, p.m.lmat, vv, work, lane);
            ncall++;
            if (lcur > loglstar_) done = true;
        }
        __syncwarp();
        for (int i = lane; i < n; i += 32) { p.u[q * n + i] = uu[i]; p.v[q * n + i] = vv[i]; }
        if (lane == 0) { p.logl[q] = lcur; p.ncall[q] = ncall; p.nprop[q] = nprop; p.flags[q] = fl; }
        __syncwarp();
    }
}

// host Philox4x32-10 (same block function as the device's curand_Philox4x32_10), for the resampling indices of a
// bootstrap realisation: one uniform vector event of the B2N stream (seed, chain), element e -> floor(U_e * N)
static inline void fr_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
    for (int r = 0; r < 10; r++) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
static inline double fr_u52(uint32_t a, uint32_t b) {
    return ((double)(a >> 6) * 67108864.0 + (double)(b >> 6) + 0.5) * 0x1p-52;
}

static int friends_dev_in(b2n_ctx* ctx, DevBuf& buf, const void* src, size_t bytes, const double** dev) {
    const void* d;
    B2N_TRY(b2n_in(ctx, buf, src, bytes, &d));
    *dev = (const double*)d;
    return B2N_OK;
}

extern "C" {

int b2n_friends_update(b2n_ctx* ctx, const double* points, int64_t N, int32_t n, int32_t kind, int32_t use_clustering,
                       const double* am_prev, int32_t nboot, uint64_t seed, uint64_t chain0, double* cov, double* am,
                       double* axes, double* axes_inv, double* logvol, double* radius, int32_t* nclusters) {
    if (!ctx || !points || N < 2 || n < 1 || (kind != 0 && kind != 1) || nboot < 0) return B2N_ERR_ARG;
    if (use_clustering && !am_prev) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    const int ld = n | 1, half = ((n + 1) & ~1) >> 1;
    const size_t met_smem = (size_t)(2 * half + 4 * n + 32 + 2 * n * ld) * sizeof(double);
    if (met_smem > (size_t)ctx->max_smem_optin) return b2n_fail(ctx, B2N_ERR_UNSUPPORTED, "ndim too large for the friends bounds (n <= ~117)");
    if (N > (1 << 20)) return b2n_fail(ctx, B2N_ERR_UNSUPPORTED, "too many points for the friends bounds");
    cudaStream_t st = ctx->stream;
    const size_t nn = (size_t)n * n;
    const double* dP;
    B2N_TRY(friends_dev_in(ctx, ctx->in0, points, (size_t)N * n * sizeof(double), &dP));
    B2N_TRY(b2n_func_smem(ctx, (const void*)(friends_metric_kernel), (size_t)(met_smem)));
    // scratch: [metric out 3nn | scal 2 | y N*n | over N*n | dist N | rmax 1]
    const size_t words = 3 * nn + 2 + 2 * (size_t)N * n + (size_t)N + 2;
    B2N_CUDA(ctx, ctx->out0.ensure(words * sizeof(double)));
    double* dmet = ctx->out0.as<double>();
    double* dscal = dmet + 3 * nn;
    double* dy = dscal + 2;
    double* dover = dy + (size_t)N * n;
    double* ddist = dover + (size_t)N * n;
    double* drmax = ddist + N;
    const unsigned wgrid = (unsigned)(((size_t)N * 32 + 255) / 256);
    int ncl = 1;
    const double* dcovsrc = dP;         // block whose np.cov is the new covariance
    if (use_clustering) {
        // ---- 1. clusters under the current metric: y = x @ T with T T^T = am_prev (T = sqrtm(am_prev))
        const double* dam;
        B2N_TRY(friends_dev_in(ctx, ctx->in1, am_prev, nn * sizeof(double), &dam));
        friends_metric_kernel<<<1, 1024, met_smem, st>>>(dam, n, ld, dmet, dscal);     // out[nn..2nn) = sqrtm(am_prev)
        B2N_LAUNCH_CHECK(ctx);
        friends_transform_kernel<<<wgrid, 256, 0, st>>>(dP, (int)N, n, dmet + nn, dy);
        B2N_LAUNCH_CHECK(ctx);
        const int W = (int)((N + 31) / 32);
        B2N_CUDA(ctx, ctx->out1.ensure((size_t)N * W * sizeof(uint32_t) + (size_t)(2 * N + 4) * sizeof(int)));
        uint32_t* dadj = ctx->out1.as<uint32_t>();
        int* dl0 = reinterpret_cast<int*>(dadj + (size_t)N * W);
        int* dl1 = dl0 + N;
        int* dchg = dl1 + N;
        friends_adj_kernel<<<(unsigned)(((size_t)N * W + 255) / 256), 256, 0, st>>>(dy, (int)N, n, W, dadj);
        B2N_LAUNCH_CHECK(ctx);
        std::vector<int> lab(N);
        for (int64_t i = 0; i < N; i++) lab[i] = (int)i;
        B2N_CUDA(ctx, cudaMemcpyAsync(dl0, lab.data(), (size_t)N * sizeof(int), cudaMemcpyHostToDevice, st));
        int* hchg = reinterpret_cast<int*>(ctx->pinned);
        int* lin = dl0;
        int* lout = dl1;
        for (int sweep = 0; sweep < (int)N + 4; sweep += 4) {
            B2N_CUDA(ctx, cudaMemsetAsync(dchg, 0, sizeof(int), st));
            for (int s4 = 0; s4 < 4; s4++) {
                friends_label_kernel<<<wgrid, 256, 0, st>>>(dadj, (int)N, W, lin, lout, dchg);
                B2N_LAUNCH_CHECK(ctx);
                std::swap(lin, lout);
            }
            B2N_CUDA(ctx, cudaMemcpyAsync(hchg, dchg, sizeof(int), cudaMemcpyDeviceToHost, st));
            B2N_CUDA(ctx, cudaStreamSynchronize(st));
            if (!*hchg) break;
        }
        B2N_CUDA(ctx, b2n_copy_sync(ctx, lab.data(), lin, (size_t)N * sizeof(int), cudaMemcpyDeviceToHost));
        // ---- clusters as segments of a permutation (ordered by root label = smallest member, members in index order)
        std::vector<int> order(N);
        for (int64_t i = 0; i < N; i++) order[i] = (int)i;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return lab[a] < lab[b]; });
        std::vector<int2> seg;
        for (int64_t i = 0; i < N;) {
            int64_t j = i;
            while (j < N && lab[order[j]] == lab[order[i]]) j++;
            seg.push_back(make_int2((int)i, (int)(j - i)));
            i = j;
        }
        ncl = (int)seg.size();
        if (ncl > 1) {          // re-centre every cluster on its own mean (:979-993)
            const void *dperm, *dseg;
            B2N_TRY(b2n_in_host(ctx, ctx->work0, order.data(), (size_t)N * sizeof(int), &dperm));
            B2N_TRY(b2n_in_host(ctx, ctx->work1, seg.data(), seg.size() * sizeof(int2), &dseg));
            friends_center_kernel<<<ncl, 256, (size_t)n * sizeof(double), st>>>(dP, n, (const int*)dperm, (const int2*)dseg, dover);
            B2N_LAUNCH_CHECK(ctx);
            dcovsrc = dover;
        }
    }
    if (nclusters) *nclusters = ncl;
    // ---- np.cov(block, ddof = 1): the node kernels on the block as one node
    BoundWork w;
    B2N_TRY(b2n_boundwork_init(ctx, w, dcovsrc, N, n, 1));
    B2N_TRY(b2n_init_identity_perm(w));
    B2N_TRY(b2n_node_moments(w, (int)N));
    // ---- 2. metric from the eigen-decomposition of the covariance
    friends_metric_kernel<<<1, 1024, met_smem, st>>>(w.na.covraw, n, ld, dmet, dscal);
    B2N_LAUNCH_CHECK(ctx);
    // ---- 3. radius
    friends_transform_kernel<<<wgrid, 256, 0, st>>>(dP, (int)N, n, dmet + 2 * nn, dy);
    B2N_LAUNCH_CHECK(ctx);
    double r = 0.0;
    if (nboot == 0) {
        friends_nn_kernel<<<wgrid, 256, 0, st>>>(dy, (int)N, n, kind, nullptr, nullptr, ddist);
        B2N_LAUNCH_CHECK(ctx);
        friends_max_kernel<<<1, 1024, 0, st>>>(ddist, (int)N, drmax);
        B2N_LAUNCH_CHECK(ctx);
        B2N_CUDA(ctx, cudaMemcpyAsync(&r, drmax, sizeof(double), cudaMemcpyDeviceToHost, st));
        B2N_CUDA(ctx, cudaStreamSynchronize(st));
    } else {
        B2N_CUDA(ctx, ctx->out2.ensure((size_t)2 * N));
        unsigned char* dmask = ctx->out2.as<unsigned char>();
        unsigned char* dwant = dmask + N;
        std::vector<unsigned char> in_bag(N), oob(N);
        for (int b = 0; b < nboot; b++) {
            const uint64_t chain = chain0 + (uint64_t)b;
            std::fill(in_bag.begin(), in_bag.end(), 0);
            for (int64_t e = 0; e < N; e += 2) {
                uint32_t o[4];
                fr_philox((uint32_t)(e >> 1), 0u, (uint32_t)chain, (uint32_t)(chain >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), o);
                int64_t i0 = (int64_t)(fr_u52(o[0], o[1]) * (double)N);
                in_bag[std::min<int64_t>(i0, N - 1)] = 1;
                if (e + 1 < N) {
                    int64_t i1 = (int64_t)(fr_u52(o[2], o[3]) * (double)N);
                    in_bag[std::min<int64_t>(i1, N - 1)] = 1;
                }
            }
            int64_t n_in = 0;                           // _bootstrap_points (:1607-1614): at least two in, one out
            for (int64_t i = 0; i < N; i++) n_in += in_bag[i];
            if (n_in < 2) in_bag[0] = in_bag[1] = 1;
            if (n_in > N - 1) in_bag[0] = 0;
            for (int64_t i = 0; i < N; i++) oob[i] = in_bag[i] ? 0 : 1;
            B2N_CUDA(ctx, cudaMemcpyAsync(dmask, in_bag.data(), (size_t)N, cudaMemcpyHostToDevice, st));
            B2N_CUDA(ctx, cudaMemcpyAsync(dwant, oob.data(), (size_t)N, cudaMemcpyHostToDevice, st));
            friends_nn_kernel<<<wgrid, 256, 0, st>>>(dy, (int)N, n, kind, dmask, dwant, ddist);
            B2N_LAUNCH_CHECK(ctx);
            friends_max_kernel<<<1, 1024, 0, st>>>(ddist, (int)N, drmax);
            B2N_LAUNCH_CHECK(ctx);
            double rb = 0.0;
            B2N_CUDA(ctx, cudaMemcpyAsync(&rb, drmax, sizeof(double), cudaMemcpyDeviceToHost, st));
            B2N_CUDA(ctx, cudaStreamSynchronize(st));
            r = std::max(r, rb);
        }
    }
    if (!(r > 0.0) || !(r < INFINITY)) return b2n_fail(ctx, B2N_ERR_SINGULAR, "friends radius is zero or not finite (coincident points)");
    // ---- 4. rescale by the radius, log-volume
    double scal[2];
    B2N_CUDA(ctx, cudaMemcpyAsync(scal, dscal, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    B2N_CUDA(ctx, cudaStreamSynchronize(st));
    friends_scale_kernel<<<64, 256, 0, st>>>(w.na.covraw, nn, r * r);
    friends_scale_kernel<<<64, 256, 0, st>>>(dmet, nn, 1.0 / (r * r));
    friends_scale_kernel<<<64, 256, 0, st>>>(dmet + nn, nn, r);
    friends_scale_kernel<<<64, 256, 0, st>>>(dmet + 2 * nn, nn, 1.0 / r);
    ctx->launches += 4;
    B2N_CUDA(ctx, cudaGetLastError());
    const cudaMemcpyKind ok = ctx->ptr_mode == B2N_PTR_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    if (cov) B2N_CUDA(ctx, cudaMemcpyAsync(cov, w.na.covraw, nn * sizeof(double), ok, st));
    if (am) B2N_CUDA(ctx, cudaMemcpyAsync(am, dmet, nn * sizeof(double), ok, st));
    if (axes) B2N_CUDA(ctx, cudaMemcpyAsync(axes, dmet + nn, nn * sizeof(double), ok, st));
    if (axes_inv) B2N_CUDA(ctx, cudaMemcpyAsync(axes_inv, dmet + 2 * nn, nn * sizeof(double), ok, st));
    B2N_CUDA(ctx, cudaStreamSynchronize(st));
    const double pref = kind == 0 ? (n * log(2.0) + n * lgamma(1.5) - lgamma(n / 2.0 + 1.0)) : n * log(2.0);   // :761, :1027
    if (logvol) *logvol = pref - 0.5 * (scal[0] - 2.0 * n * log(r));
    if (radius) *radius = r;
    return B2N_OK;
}

int b2n_friends_set(b2n_ctx* ctx, int32_t kind, const double* ctrs, int64_t N, int32_t n, const double* axes,
                    const double* axes_inv) {
    if (!ctx || !ctrs || !axes || !axes_inv || N < 1 || n < 1 || (kind != 0 && kind != 1)) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    FriendsState* f = friends_of(ctx);
    const size_t nn = (size_t)n * n;
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    B2N_CUDA(ctx, f->ctrs.ensure((size_t)N * n * sizeof(double)));
    B2N_CUDA(ctx, f->ctrs_t.ensure((size_t)N * n * sizeof(double)));
    B2N_CUDA(ctx, f->axes.ensure(nn * sizeof(double)));
    B2N_CUDA(ctx, f->axes_inv.ensure(nn * sizeof(double)));
    const cudaMemcpyKind k = ctx->ptr_mode == B2N_PTR_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    B2N_CUDA(ctx, cudaMemcpyAsync(f->ctrs.p, ctrs, (size_t)N * n * sizeof(double), k, ctx->stream));
    B2N_CUDA(ctx, cudaMemcpyAsync(f->axes.p, axes, nn * sizeof(double), k, ctx->stream));
    B2N_CUDA(ctx, cudaMemcpyAsync(f->axes_inv.p, axes_inv, nn * sizeof(double), k, ctx->stream));
    friends_transform_kernel<<<(unsigned)(((size_t)N * 32 + 255) / 256), 256, 0, ctx->stream>>>(
        f->ctrs.as<double>(), (int)N, n, f->axes_inv.as<double>(), f->ctrs_t.as<double>());
    B2N_LAUNCH_CHECK(ctx);
    f->kind = kind; f->N = (int)N; f->n = n;
    return b2n_finish(ctx);
}

int b2n_friends_overlap(b2n_ctx* ctx, const double* x, int64_t M, int32_t n, int32_t* q) {
    if (!ctx || !x || !q || M < 0) return B2N_ERR_ARG;
    FriendsState* f = friends_of(ctx);
    if (f->N < 1 || f->n != n) return b2n_fail(ctx, B2N_ERR_ARG, "no resident friends bound of this dimension (b2n_friends_set)");
    if (M == 0) return B2N_OK;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    const void* dx;
    void* dq;
    B2N_TRY(b2n_in(ctx, ctx->in0, x, (size_t)M * n * sizeof(double), &dx));
    B2N_TRY(b2n_out(ctx, ctx->out3, q, (size_t)M * sizeof(int), &dq));
    const int wpb = 4;
    const size_t smem = (size_t)wpb * n * sizeof(double);
    friends_overlap_kernel<<<(unsigned)std::min<int64_t>((M + wpb - 1) / wpb, 148 * 16), wpb * 32, smem, ctx->stream>>>(
        (const double*)dx, M, n, f->kind, f->ctrs_t.as<double>(), f->N, f->axes_inv.as<double>(), (int*)dq);
    B2N_LAUNCH_CHECK(ctx);
    B2N_TRY(b2n_out_done(ctx, q, dq, (size_t)M * sizeof(int)));
    return b2n_finish(ctx);
}

int b2n_friends_unif_batch(b2n_ctx* ctx, const b2n_chain_args* a, double* u, double* v, double* logl, int32_t* ncall,
                           int32_t* nprop, uint32_t* flags) {
    if (!ctx || !a || !u || !v || !logl || !ncall || !nprop || !flags) return B2N_ERR_ARG;
    FriendsState* f = friends_of(ctx);
    const int draw_only = (a->reserved & B2N_OPT_DRAW_ONLY) ? ((a->reserved & B2N_OPT_DRAW_MIXTURE) ? 3 : 1) : 0;
    B2nModel m;
    memset(&m, 0, sizeof(m));
    m.ndim = a->ndim;
    m.like_kind = B2N_LIKE_EGGBOX;
    if (!draw_only) {
        if (a->model_id < 0 || a->model_id >= (int)ctx->models.size()) return B2N_ERR_ARG;
        m = ctx->models[a->model_id];
    }
    const int n = a->ndim;
    const int64_t Q = a->nchain;
    if (f->N < 1 || f->n != n || n != m.ndim || a->ncdim != n || Q < 0)
        return b2n_fail(ctx, B2N_ERR_ARG, "friends sampling needs a resident friends bound with ncdim == ndim");
    if (Q == 0) return B2N_OK;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    const void* dfl_in = nullptr;
    std::vector<uint32_t> fl;
    if (a->dimflags) {
        fl.assign(a->dimflags, a->dimflags + n);
        B2N_TRY(b2n_in_host(ctx, ctx->in3, fl.data(), fl.size() * sizeof(uint32_t), &dfl_in));
    }
    FriendsUnifParams p;
    p.m = m; p.n = n; p.N = f->N; p.kind = f->kind; p.draw_only = draw_only;
    p.ctrs = f->ctrs.as<double>(); p.ctrs_t = f->ctrs_t.as<double>(); p.axes = f->axes.as<double>(); p.axes_inv = f->axes_inv.as<double>();
    p.dimflags = (const uint32_t*)dfl_in; p.loglstar = a->loglstar; p.seed = a->seed; p.chain0 = a->chain0; p.Q = Q;
    p.dyn = nullptr;
    void *du, *dv, *dl, *dnc, *dnp, *dfl;
    B2N_TRY(b2n_out(ctx, ctx->out0, u, (size_t)Q * n * sizeof(double), &du));
    B2N_TRY(b2n_out(ctx, ctx->out1, v, (size_t)Q * n * sizeof(double), &dv));
    B2N_TRY(b2n_out(ctx, ctx->out2, logl, (size_t)Q * sizeof(double), &dl));
    B2N_TRY(b2n_out(ctx, ctx->out3, ncall, (size_t)Q * sizeof(int), &dnc));
    B2N_TRY(b2n_out(ctx, ctx->out4, nprop, (size_t)Q * sizeof(int), &dnp));
    B2N_TRY(b2n_out(ctx, ctx->out6, flags, (size_t)Q * sizeof(uint32_t), &dfl));
    p.u = (double*)du; p.v = (double*)dv; p.logl = (double*)dl; p.ncall = (int*)dnc; p.nprop = (int*)dnp; p.flags = (uint32_t*)dfl;
    const int threads = 128, wpb = threads / 32;
    const size_t smem = (size_t)wpb * 5 * n * sizeof(double);
    if (smem > (size_t)ctx->max_smem_optin) return b2n_fail(ctx, B2N_ERR_UNSUPPORTED, "ndim too large for the friends kernel");
    const int64_t blocks = (Q + wpb - 1) / wpb;
#define CALL(L)                                                                                                   \
    if (smem > 48 * 1024)                                                                                         \
        B2N_TRY(b2n_func_smem(ctx, (const void*)(friends_unif_kernel<L>), (size_t)(smem))); \
    friends_unif_kernel<L><<<(unsigned)blocks, threads, smem, ctx->stream>>>(p);
    B2N_DISPATCH_LIKE(m.like_kind, CALL)
#undef CALL
    B2N_LAUNCH_CHECK(ctx);
    B2N_TRY(b2n_out_done(ctx, u, du, (size_t)Q * n * sizeof(double)));
    B2N_TRY(b2n_out_done(ctx, v, dv, (size_t)Q * n * sizeof(double)));
    B2N_TRY(b2n_out_done(ctx, logl, dl, (size_t)Q * sizeof(double)));
    B2N_TRY(b2n_out_done(ctx, ncall, dnc, (size_t)Q * sizeof(int)));
    B2N_TRY(b2n_out_done(ctx, nprop, dnp, (size_t)Q * sizeof(int)));
    B2N_TRY(b2n_out_done(ctx, flags, dfl, (size_t)Q * sizeof(uint32_t)));
    return b2n_finish(ctx);
}

}  // extern "C"

// ---- friends mode of the device-resident rounds (b2n_ns.cu) -------------------------------------------------------
int b2n_friends_transform_dev(b2n_ctx* ctx, const double* x, int N, int n, const double* T, double* y) {
    friends_transform_kernel<<<(unsigned)(((size_t)N * 32 + 255) / 256), 256, 0, ctx->stream>>>(x, N, n, T, y);
    B2N_LAUNCH_CHECK(ctx);
    return B2N_OK;
}

int b2n_friends_rescale_dev(b2n_ctx* ctx, int n, double* cov, double* am, double* axes, double* axes_inv, double f) {
    const size_t nn = (size_t)n * n;
    friends_rescale_kernel<<<(unsigned)std::min<size_t>((nn + 255) / 256, 64), 256, 0, ctx->stream>>>(
        cov, am, axes, axes_inv, nn, f, pow(f, 2.0));
    B2N_LAUNCH_CHECK(ctx);
    return B2N_OK;
}

// One device-paced launch of friends_unif_kernel for the K chains of a round: the centres are the run's live set as it
// stands (the reference re-points bound.ctrs = live_u before every proposal, sampler.py:479-482), ctrs_t its rows
// times axes_inv, kept current by the round's commit kernel.  Threshold and chain ids come from ctx->dyn.
int b2n_friends_unif_dev(b2n_ctx* ctx, const b2n_chain_args* a, int N, int kind, const double* ctrs, const double* ctrs_t,
                         const double* axes, const double* axes_inv, double* u, double* v, double* logl, int32_t* ncall,
                         int32_t* nprop, uint32_t* flags) {
    if (!ctx->dyn.active || ctx->ptr_mode != B2N_PTR_DEVICE) return b2n_fail(ctx, B2N_ERR_ARG, "b2n_friends_unif_dev: device-paced launches only");
    ctx->dyn.cpc = 1;
    if (ctx->dyn.plan_only) return B2N_OK;
    if (a->model_id < 0 || a->model_id >= (int)ctx->models.size()) return B2N_ERR_ARG;
    const B2nModel m = ctx->models[a->model_id];
    const int n = a->ndim;
    const int64_t Q = a->nchain;
    if (n != m.ndim || a->ncdim != n || Q < 1 || N < 1) return B2N_ERR_ARG;
    const void* dfl_in = nullptr;
    std::vector<uint32_t> fl;
    if (a->dimflags) {
        fl.assign(a->dimflags, a->dimflags + n);
        B2N_TRY(b2n_in_host(ctx, ctx->in3, fl.data(), fl.size() * sizeof(uint32_t), &dfl_in));
    }
    FriendsUnifParams p;
    p.m = m; p.n = n; p.N = N; p.kind = kind; p.draw_only = 0;
    p.ctrs = ctrs; p.ctrs_t = ctrs_t; p.axes = axes; p.axes_inv = axes_inv;
    p.dimflags = (const uint32_t*)dfl_in; p.loglstar = a->loglstar; p.seed = a->seed; p.chain0 = a->chain0; p.Q = Q;
    p.u = u; p.v = v; p.logl = logl; p.ncall = ncall; p.nprop = nprop; p.flags = flags;
    p.dyn = ctx->dyn.dev;
    const int threads = 128, wpb = threads / 32;
    const size_t smem = (size_t)wpb * 5 * n * sizeof(double);
    if (smem > (size_t)ctx->max_smem_optin) return b2n_fail(ctx, B2N_ERR_UNSUPPORTED, "ndim too large for the friends kernel");
    const int64_t blocks = (Q + wpb - 1) / wpb;
#define CALL(L)                                                                                                   \
    if (smem > 48 * 1024)                                                                                         \
        B2N_TRY(b2n_func_smem(ctx, (const void*)(friends_unif_kernel<L>), (size_t)(smem))); \
    friends_unif_kernel<L><<<(unsigned)blocks, threads, smem, ctx->stream>>>(p);
    B2N_TIME_BEGIN(ctx);
    B2N_DISPATCH_LIKE(m.like_kind, CALL)
    B2N_TIME_END(ctx);
#undef CALL
    B2N_LAUNCH_CHECK(ctx);
    return B2N_OK;            // the commit kernel of the round folds the flags (draw limit: 0x80000000)
}
