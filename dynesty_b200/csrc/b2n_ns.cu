// b2n_ns.cu -- device-resident nested-sampling rounds ("replace the K worst live points per
// launch", SURVEY.md 8(f)1).  Part of libb200nest.so (C ABI: include/b200nest.h, b2n_ns_*).
//
// What it replaces.  The reference's master loop (sampler.py:1040-1212) removes ONE worst live
// point per iteration and obtains its replacement from `_new_point` (:732-778), which pops a
// queue that `_fill_queue` (:676-717) fills with `queue_size` proposals evolved at the threshold
// of fill time.  With a queue, an entry is kept only if it still beats the CURRENT threshold: for
// chains that stay correlated with their start point (rwalk at 50-D) that filter selects the
// offspring of the best live points and biases logZ (DESIGN.md 9.4) -- and every iteration costs
// a host round trip.  A round here removes the K lowest live points AT ONCE (threshold = the
// K-th lowest logl), evolves K chains from uniformly chosen survivors at that threshold and puts
// every chain end point into a freed slot: no filter, hence no selection effect, and every
// proposal is used.  Between the removals the number of live points falls N, N-1, .. N-K+1,
// which the evidence quadrature accounts for exactly as the reference does for a shrinking
// live set (sampler.py:780-914 / utils.py:1411-1467): ln X decreases by ln((m+1)/m) at a dead
// point that had m live points.
//
// One round = three launches on the ctx stream, no host synchronisation in between:
//   ns_propose_kernel  termination test (sampler.py:1095-1120) on the sorted live log-likelihoods (kept
//                      sorted across rounds: one bitonic sort at start-up, then a K-into-(N-K) merge
//                      per round in the commit kernel), pick K start rows among the survivors and their
//                      ellipsoids (propose_live :469-491, get_random_axes bounding.py:726-731),
//                      `bound.contains` of every start (:485-489), build the per-CTA worklist of
//                      the chain kernel, write the round's B2nDyn
//   chain kernel       rwalk / rslice / slice / unif (b2n_rwalk.cu, b2n_slice.cu, b2n_unif.cu), device-paced
//   ns_commit_kernel   dead-point records, evidence increment (utils.py:1470-1492), scatter of the
//                      chain end points into the freed slots, tuning of the proposal scale
//                      (internal_samplers.py:460-493, 1209-1239), bound-update-due test
//                      (sampler.py:625-674)
// A stop condition (done / bound update due / start outside the bound / dead buffer full) sets a
// flag in HBM; the remaining enqueued rounds return at once and the host picks the flag up at its
// next status read.
#include "b2n_device.cuh"
#include <algorithm>
#include <math_constants.h>

#define B2N_NS_DRIVER_CHAIN 0x4000000000000000ULL   // Philox chain id space of the round driver
// Philox chain id space of the bootstrap realisations of the friends bounds' device updates (b2n_ns_update_friends):
// realisation b of an update made at round r is the chain B2N_NS_FRIENDS_BOOT_CHAIN + (r << 8) + b, b < 256 --
// disjoint from the live-point initialisation (2^61 + i), the round driver (2^62 + r) and the chains (chain0 + r K + c)
#define B2N_NS_FRIENDS_BOOT_CHAIN 0x6000000000000000ULL
#define B2N_NS_FRIENDS_MAX_BOOT 255
#define B2N_NS_THREADS 1024

struct NsScalars {
    long long it, ncall, ncall_last_update, round;
    double logvol, logz, loglstar, lmax, scale, delta_logz;
    long long hist_a, hist_b;
    int done, need_bound, doubling, error;
    int parity, pad0;          // which of the two (key, row) buffer pairs holds the current sorted order
    int phase, pending;        // phase 0: unit-cube rounds (no bound yet), 1: bounded rounds.  pending: a round
                               // has been proposed (its chains are in flight) and waits for its commit
};

struct NsDev {
    int N, n, nc, K, Kell, cpc, strict, sampler, Npad, Kpad, threads;
    double dlogz, facc, first_min_eff, logl_max;
    long long maxiter, maxcall, update_interval, dead_cap, first_min_ncall, it0;
    unsigned long long seed, chain0;
    double *live_u, *live_v, *live_logl;
    double *dead_u, *dead_v, *dead_logl, *dead_logvol;
    int* dead_ncall;
    NsScalars* sc;
    B2nDyn* dyn;
    int* sidx;          // live rows sorted by (logl, row) ascending -- maintained across rounds
    double* skey;       // their logl
    int* tidx;          // merge scratch
    double* tkey;
    double* u0;         // K x n start points of the round
    int* order;         // chain worklist
    int3* cta;
    double *o_u, *o_v, *o_logl;
    int *o_i0, *o_i1, *o_ncall;
    uint32_t* o_flags;
    const double *ctrs, *ams, *logvols;      // resident bound
    // friends mode (RadFriends / SupFriends, b2n_ns_update_friends / b2n_ns_set_friends): one ball / cube of common
    // shape around every live point.  Kell = 1 and no contains test (a start point is a live point, hence a centre).
    int friends, pad1;
    const double* fr_axes_inv;   // uniform sampler only: the commit refreshes the replaced rows of fr_ctrs_t =
    double* fr_ctrs_t;           // live_u @ axes_inv (the transformed centres friends_unif_kernel counts q with)
};

struct b2n_ns {
    b2n_ns_config cfg;
    std::vector<uint8_t> dimflags;
    bool has_flags = false;
    NsDev d;
    long long dead_cap = 0;
    std::vector<void*> allocs;
    void* dead_alloc[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    int phase = 1;                     // host copy of NsScalars::phase (transitions are host-mediated)
    // CUDA graph of B2N_NS_GRAPH_ROUNDS rounds ([commit+propose | chains] x G): every per-round argument of these
    // kernels lives in HBM (B2nDyn, NsScalars), so the launch sequence is STATIC and a block of rounds can be one
    // cudaGraphLaunch instead of 2 G kernel launches.  Re-captured when anything baked into the kernel arguments
    // changes.  Opt-in, see b2n_ns_run.
    cudaGraphExec_t gexec = nullptr;
    unsigned long long gkey = 0, warm_key = 0;
    bool active = false;               // between b2n_ns_create and b2n_ns_destroy.  The device allocations OUTLIVE a run
                                       // (released by b2n_free, or by a b2n_ns_create of another shape): cudaMalloc /
                                       // cudaFree synchronise the whole device, which would stall every other replica
                                       // running on this GPU (dynesty_b200/replicas.py) once per run
    // device copy of the bound built by b2n_ns_update_bound (Kmax ellipsoids of dimension nc)
    int Kmax = 0, bK = 0;
    double *bd_ctrs = nullptr, *bd_covs = nullptr, *bd_ams = nullptr, *bd_axes = nullptr, *bd_axlens = nullptr,
           *bd_logvols = nullptr, *bd_points = nullptr;
    std::vector<double> bd_hlogvols;
    // friends mode: the run's RadFriends / SupFriends bound (n x n each), allocated by the first friends entry point.
    // fr_ready: a bound exists (fit or adopted); fr_am is the am_prev of the next update.
    bool friends = false, fr_ready = false;
    int fr_kind = 0, fr_ncl = 0;
    double fr_logvol = 0.0, fr_radius = 0.0;
    double *fr_cov = nullptr, *fr_am = nullptr, *fr_axes = nullptr, *fr_axinv = nullptr, *fr_ctrs_t = nullptr;
    unsigned long long fr_serial = 0;  // ctx->bound_serial right after this run made its axes the resident bound
};

__device__ __forceinline__ double dev_logaddexp(double a, double b) {
    const double hi = fmax(a, b), lo = fmin(a, b);
    if (lo == -CUDART_INF) return hi;
    return hi + log1p(exp(lo - hi));
}

// ---------------------------------------------------------------------------------------------
// full sort of the live log-likelihoods (start-up only): bitonic over (logl, row), one CTA
__global__ void __launch_bounds__(B2N_NS_THREADS, 1) ns_sort_kernel(const NsDev s) {
    extern __shared__ __align__(16) unsigned char ns_smem[];
    const int tid = threadIdx.x, nth = blockDim.x;
    const int N = s.N, Npad = s.Npad;
    double* key = reinterpret_cast<double*>(ns_smem);
    int* idx = reinterpret_cast<int*>(key + Npad);
    for (int i = tid; i < Npad; i += nth) {
        key[i] = i < N ? s.live_logl[i] : CUDART_INF;     // padding (+inf, row >= N) sorts last
        idx[i] = i;
    }
    __syncthreads();
    for (int k = 2; k <= Npad; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < (Npad >> 1); t += nth) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const int l = i | j;
                const bool asc = (i & k) == 0;
                const double ka = key[i], kb = key[l];
                const int ia = idx[i], ib = idx[l];
                const bool gt = ka > kb || (ka == kb && ia > ib);
                if (gt == asc) { key[i] = kb; key[l] = ka; idx[i] = ib; idx[l] = ia; }
            }
            __syncthreads();
        }
    }
    for (int i = tid; i < N; i += nth) { s.sidx[i] = idx[i]; s.skey[i] = key[i]; }
}

extern __shared__ __align__(16) unsigned char ns_smem[];

__device__ __forceinline__ void ns_propose_body(const NsDev& s) {
    const int tid = threadIdx.x, nth = blockDim.x, warp = tid >> 5, lane = tid & 31;
    NsScalars* sc = s.sc;
    if (sc->done || sc->need_bound) {
        if (tid == 0) s.dyn->skip = 1;
        return;
    }
    const int N = s.N, K = s.K, n = s.n, nc = s.nc;
    double* dvec = reinterpret_cast<double*>(ns_smem);       // (warps) x nc
    double* cum = dvec + (nth >> 5) * nc;                    // Kell
    int* start = reinterpret_cast<int*>(cum + ((s.Kell + 1) & ~1));   // K
    int* ell = start + K;                                    // K
    int* cnt = ell + K;                                      // Kell + 1
    const int par = sc->parity;                              // current sorted order: ascending by (logl, row)
    const double* key = par ? s.tkey : s.skey;
    const int* idx = par ? s.tidx : s.sidx;
    __shared__ int s_flag, s_bad, s_first;
    if (tid == 0) { s_flag = 0; s_bad = 0; s_first = K; }
    __syncthreads();
    // ---- termination (sampler.py:1095-1120) and capacity
    if (tid == 0) {
        const double lmax = key[N - 1];
        const double delta = dev_logaddexp(0.0, lmax + sc->logvol - sc->logz);
        sc->lmax = lmax;
        sc->delta_logz = delta;
        // (maxiter is tested per round: a run may overshoot it by up to batch - 1 iterations.  logl_max: the stop
        //  of a dynamic-sampler batch, dynamicsampler.py:1338-1345 -- the worst live point has left the range)
        if (delta < s.dlogz || sc->it >= s.maxiter || sc->ncall >= s.maxcall || key[0] == lmax || key[0] > s.logl_max) {
            sc->done = 1;
            s_flag = 1;
        } else if (sc->it + K > s.dead_cap) {
            sc->need_bound = 3;                             // dead buffer full: the host grows it
            s_flag = 1;
        } else {
            // start rows must have logl STRICTLY above the threshold key[K-1] (sampler.py:471: live_logl > loglstar):
            // with ties at the threshold (plateau likelihoods, a stuck chain duplicating its start) the sorted
            // suffix begins later than K.  Binary search for the first key > threshold.
            const double thr = key[K - 1];
            int lo = K, hi = N;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (key[mid] > thr) hi = mid; else lo = mid + 1;
            }
            s_first = lo;
            if (lo >= N) {                                   // no live point above the threshold: plateau
                sc->done = 1;
                sc->error = B2N_ERR_PLATEAU;
                s_flag = 1;
            }
        }
        if (s_flag) s.dyn->skip = 1;
    }
    __syncthreads();
    if (s_flag) return;
    if (s.sampler == 3 || sc->phase == 0) {   // uniform / unit-cube sampler: the chains draw themselves -- no start rows
        if (tid == 0) {
            B2nDyn* dy = s.dyn;
            dy->loglstar = key[K - 1];
            dy->scale = sc->scale;
            dy->chain0 = s.chain0 + (unsigned long long)sc->round * (unsigned long long)K;
            dy->ncta = 0;
            dy->doubling = 0;
            dy->skip = 0;
            sc->pending = 1;
        }
        return;
    }
    // ---- start rows among the survivors, ellipsoid of every chain
    ChainRng g;
    g.init(s.seed, B2N_NS_DRIVER_CHAIN + (unsigned long long)sc->round);
    if (s.Kell > 1 && tid == 0) {                           // volume-weighted pick: cumulative probabilities
        double m = s.logvols[0];
        for (int k = 1; k < s.Kell; k++) m = fmax(m, s.logvols[k]);
        double tot = 0.0;
        for (int k = 0; k < s.Kell; k++) tot += exp(s.logvols[k] - m);
        const double lv = m + log(tot);
        double c = 0.0;
        for (int k = 0; k < s.Kell; k++) { c += exp(s.logvols[k] - lv); cum[k] = c; }
    }
    __syncthreads();
    const int first = s_first, nsurv = N - first;
    for (int c = tid; c < K; c += nth) {
        g.tick = 0;
        const double U = rng_uniform_elem(g, c);
        int sidx = (int)(U * (double)nsurv);
        sidx = sidx < nsurv - 1 ? sidx : nsurv - 1;
        start[c] = idx[first + sidx];
        int e = 0;
        if (s.Kell > 1) {
            g.tick = 1;
            const double U2 = rng_uniform_elem(g, c);
            while (e < s.Kell - 1 && cum[e] < U2) e++;       // np.searchsorted(cumsum, U), clipped
        }
        ell[c] = e;
    }
    __syncthreads();
    // ---- bound.contains(start[:nc]) (sampler.py:485-489): a start outside forces a bound update.  Not with the
    //      friends bounds: the start is a live point, i.e. a centre of the bound (distance 0), so the forced update
    //      of sampler.py:485-489 can never fire
    for (int c = warp; c < K && !s.friends; c += (nth >> 5)) {
        const double* x = s.live_u + (size_t)start[c] * n;
        double* d = dvec + warp * nc;
        bool inside = false;
        for (int k = 0; k < s.Kell && !inside; k++) {
            const double* ctr = s.ctrs + (size_t)k * nc;
            const double* A = s.ams + (size_t)k * nc * nc;
            for (int i = lane; i < nc; i += 32) d[i] = x[i] - ctr[i];
            __syncwarp();
            double acc = 0.0;
            for (int i = lane; i < nc; i += 32) {        // A is symmetric: read it column-wise (coalesced)
                double y0 = 0.0, y1 = 0.0;
                int j = 0;
                for (; j + 1 < nc; j += 2) {
                    y0 = fma(__ldg(A + (size_t)j * nc + i), d[j], y0);
                    y1 = fma(__ldg(A + (size_t)(j + 1) * nc + i), d[j + 1], y1);
                }
                if (j < nc) y0 = fma(__ldg(A + (size_t)j * nc + i), d[j], y0);
                acc = fma(d[i], y0 + y1, acc);
            }
            acc = warp_sum(acc);
            inside = s.strict ? (acc < 1.0) : (acc <= 1.0);
            __syncwarp();
        }
        if (!inside && lane == 0) atomicOr(&s_bad, 1);
    }
    // ---- start points of the chains
    for (int e = tid; e < K * n; e += nth) {
        const int c = e / n, i = e - c * n;
        s.u0[e] = s.live_u[(size_t)start[c] * n + i];
    }
    __syncthreads();
    // ---- worklist: chains grouped by ellipsoid, groups split into equal CTAs (b2n_build_worklist)
    int ncta = 0;
    if (s.Kell == 1) {
        const int parts = (K + s.cpc - 1) / s.cpc;
        for (int c = tid; c < K; c += nth) s.order[c] = c;
        for (int i = tid; i < parts; i += nth) {
            const int lo = (int)((long long)K * i / parts), hi = (int)((long long)K * (i + 1) / parts);
            s.cta[i] = make_int3(lo, hi - lo, 0);
        }
        ncta = parts;
    } else if (tid == 0) {
        for (int k = 0; k <= s.Kell; k++) cnt[k] = 0;
        for (int c = 0; c < K; c++) cnt[ell[c] + 1]++;
        for (int k = 0; k < s.Kell; k++) cnt[k + 1] += cnt[k];
        for (int k = 0; k < s.Kell; k++) {
            const int c0 = cnt[k], c = cnt[k + 1] - c0;
            if (c == 0) continue;
            const int parts = (c + s.cpc - 1) / s.cpc;
            for (int i = 0; i < parts; i++) {
                const int lo = c0 + (int)((long long)c * i / parts), hi = c0 + (int)((long long)c * (i + 1) / parts);
                s.cta[ncta++] = make_int3(lo, hi - lo, k);
            }
        }
        // stable fill (chains of one ellipsoid keep their order); cnt[k] becomes the write cursor
        for (int c = 0; c < K; c++) s.order[cnt[ell[c]]++] = c;
    }
    if (tid == 0) {
        B2nDyn* dy = s.dyn;
        dy->loglstar = key[K - 1];
        dy->scale = sc->scale;
        dy->chain0 = s.chain0 + (unsigned long long)sc->round * (unsigned long long)K;
        dy->ncta = ncta;
        dy->doubling = sc->doubling;
        dy->skip = s_bad ? 1 : 0;
        if (s_bad) sc->need_bound = 2;                       // forced update (sampler.py:486)
        else sc->pending = 1;
    }
}

// ---------------------------------------------------------------------------------------------
// Block reductions: warp shuffles, one partial per warp in shared memory, first warp finishes.
// Fixed order (lane tree, then warp 0 over the partials): bit-reproducible for a given blockDim.
__device__ __forceinline__ double block_reduce_max(double v, double* buf) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
    v = warp_max(v);
    if (lane == 0) buf[w] = v;
    __syncthreads();
    double r = lane < nw ? buf[lane] : -CUDART_INF;
    r = warp_max(r);
    __syncthreads();
    return r;
}
__device__ __forceinline__ double block_reduce_sum(double v, double* buf) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
    v = warp_sum(v);
    if (lane == 0) buf[w] = v;
    __syncthreads();
    double r = lane < nw ? buf[lane] : 0.0;
    r = warp_sum(r);
    __syncthreads();
    return r;
}
__device__ __forceinline__ long long block_reduce_sum_ll(long long v, long long* buf) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(B2N_FULL, v, o);
    if (lane == 0) buf[w] = v;
    __syncthreads();
    long long r = lane < nw ? buf[lane] : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(B2N_FULL, r, o);
    __syncthreads();
    return r;
}

__device__ __forceinline__ void ns_commit_body(const NsDev& s) {
    if (!s.sc->pending) return;
    __shared__ double rbuf[64];
    __shared__ unsigned int s_or;
    long long* lbuf = reinterpret_cast<long long*>(rbuf);
    const int tid = threadIdx.x, nth = blockDim.x;
    NsScalars* sc = s.sc;
    const int N = s.N, K = s.K, n = s.n;
    const long long it0 = sc->it;
    const double logvol0 = sc->logvol, lprev0 = sc->loglstar;
    const int par = sc->parity;
    const double* ckey = par ? s.tkey : s.skey;      // current sorted order (read) ...
    const int* cidx = par ? s.tidx : s.sidx;
    double* nkey = par ? s.skey : s.tkey;            // ... the merged order of the next round (written)
    int* nidx = par ? s.sidx : s.tidx;
    if (tid == 0) s_or = 0u;
    __syncthreads();
    // ---- dead-point rows out, chain end points in (slot of the j-th lowest <- chain j)
    for (int e = tid; e < K * n; e += nth) {
        const int j = e / n, i = e - j * n;
        const size_t src = (size_t)cidx[j] * n + i;
        const size_t dst = (size_t)(it0 + j) * n + i;
        s.dead_u[dst] = s.live_u[src];
        s.dead_v[dst] = s.live_v[src];
        s.live_u[src] = s.o_u[e];
        s.live_v[src] = s.o_v[e];
    }
    if (s.fr_ctrs_t) {      // friends mode, uniform sampler: transformed centres of the K new rows, with the arithmetic
                            // of friends_transform_kernel (k ascending, fma) -- equal to a full re-transform bit for bit
        for (int e = tid; e < K * n; e += nth) {
            const int j = e / n, i = e - j * n;
            const double* x = s.o_u + (size_t)j * n;
            double acc = 0.0;
            for (int k = 0; k < n; k++) acc = fma(x[k], __ldg(s.fr_axes_inv + (size_t)k * n + i), acc);
            s.fr_ctrs_t[(size_t)cidx[j] * n + i] = acc;
        }
    }
    // ---- evidence: ln X_j = ln X_0 + ln((N-j)/(N+1)); trapezoid weight with dX_j = X_j / (N-j) * 1/2 ..
    double wmax = -CUDART_INF;
    long long ncall = 0, ha = 0, hb = 0;
    unsigned int fl = 0;
    for (int j = tid; j < K; j += nth) {
        const double L = ckey[j], Lp = j ? ckey[j - 1] : lprev0;
        const double lv = logvol0 + log((double)(N - j) / (double)(N + 1));
        const double w = dev_logaddexp(L, Lp) + lv + log(0.5 / (double)(N - j));
        wmax = fmax(wmax, w);
        s.dead_logl[it0 + j] = L;
        s.dead_logvol[it0 + j] = lv;
        s.dead_ncall[it0 + j] = s.o_ncall[j];
        const double lo = s.o_logl[j];
        s.live_logl[cidx[j]] = lo;
        ncall += s.o_ncall[j];
        ha += s.o_i0[j];
        hb += s.o_i1[j];
        if (s.sampler != 0 || s.sc->phase == 0) fl |= s.o_flags[j];   // rwalk writes no flags; unit-cube chains do
    }
    const double m = block_reduce_max(wmax, rbuf);
    double se = 0.0;
    for (int j = tid; j < K; j += nth) {
        const double L = ckey[j], Lp = j ? ckey[j - 1] : lprev0;
        const double lv = logvol0 + log((double)(N - j) / (double)(N + 1));
        se += exp(dev_logaddexp(L, Lp) + lv + log(0.5 / (double)(N - j)) - m);
    }
    se = block_reduce_sum(se, rbuf);
    ncall = block_reduce_sum_ll(ncall, lbuf);
    ha = block_reduce_sum_ll(ha, lbuf);
    hb = block_reduce_sum_ll(hb, lbuf);
    if (fl) atomicOr(&s_or, fl);
    __syncthreads();
    // ---- keep (skey, sidx) sorted: the K lowest were replaced, so merge the K new (logl, row) pairs
    //      into the N-K survivors (already sorted).  Comparator = (logl, row) lexicographic, a strict
    //      total order, hence position = own rank + number of elements of the OTHER list below.
    {
        const int NA = N - K, Kpad = s.Kpad;
        double* akey = reinterpret_cast<double*>(ns_smem);       // NA survivors
        double* bkey = akey + NA + (NA & 1);                      // Kpad new
        int* aidx = reinterpret_cast<int*>(bkey + Kpad);
        int* bidx = aidx + NA;
        const double thr_keep = ckey[K - 1];
        for (int i = tid; i < NA; i += nth) { akey[i] = ckey[K + i]; aidx[i] = cidx[K + i]; }
        for (int j = tid; j < Kpad; j += nth) {
            bkey[j] = j < K ? s.o_logl[j] : CUDART_INF;
            bidx[j] = j < K ? cidx[j] : 0x7fffffff;
        }
        __syncthreads();
        for (int k = 2; k <= Kpad; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = tid; t < (Kpad >> 1); t += nth) {
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                    const int l = i | j;
                    const bool asc = (i & k) == 0;
                    const double ka = bkey[i], kb = bkey[l];
                    const int ia = bidx[i], ib = bidx[l];
                    const bool gt = ka > kb || (ka == kb && ia > ib);
                    if (gt == asc) { bkey[i] = kb; bkey[l] = ka; bidx[i] = ib; bidx[l] = ia; }
                }
                __syncthreads();
            }
        }
        for (int i = tid; i < NA; i += nth) {                     // survivors: count new pairs below
            const double ka = akey[i];
            const int ia = aidx[i];
            int lo = 0, hi = K;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                const bool less = bkey[mid] < ka || (bkey[mid] == ka && bidx[mid] < ia);
                if (less) lo = mid + 1; else hi = mid;
            }
            nkey[i + lo] = ka;
            nidx[i + lo] = ia;
        }
        for (int j = tid; j < K; j += nth) {                      // new pairs: count survivors below
            const double kb = bkey[j];
            const int ib = bidx[j];
            int lo = 0, hi = NA;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                const bool less = akey[mid] < kb || (akey[mid] == kb && aidx[mid] < ib);
                if (less) lo = mid + 1; else hi = mid;
            }
            nkey[j + lo] = kb;
            nidx[j + lo] = ib;
        }
        __syncthreads();
        if (tid == 0) sc->loglstar = thr_keep;
    }
    if (tid == 0) {
        sc->logz = dev_logaddexp(sc->logz, m + log(se));
        sc->logvol = logvol0 + log((double)(N - K + 1) / (double)(N + 1));
        sc->lmax = nkey[N - 1];
        sc->parity = par ^ 1;
        sc->it = it0 + K;
        sc->ncall += ncall;
        sc->round += 1;
        sc->pending = 0;
        // ---- tune (update=True every round: the queue of the round has drained, sampler.py:757-768)
        sc->hist_a = ha;
        sc->hist_b = hb;
        if (sc->phase == 0) {                                // UnitCubeSampler: nothing to tune
            if (s_or & 0x80000000u) { sc->error = B2N_ERR_UNSUPPORTED; sc->done = 1; }   // draw limit
        } else if (s.sampler == 3) {                                // UniformBoundSampler: nothing to tune
            if (s_or & 0x40000000u) { sc->error = B2N_ERR_Q0; sc->done = 1; }            // bounding.py:570-574
            if (s_or & 0x80000000u) { sc->error = B2N_ERR_UNSUPPORTED; sc->done = 1; }   // draw limit
        } else if (s.sampler == 0) {                         // internal_samplers.py:460-493
            // The reference tunes after EVERY iteration (queue_size 1): scale *= exp((a_t - f) / (n f)) with the
            // acceptance a_t of that iteration's chain.  A round is K such iterations at one scale, i.e. the product
            // exp(K (abar - f) / (n f)); the power is capped at n so that the loop gain stays below 1 / f whatever
            // batch the caller picks.  K = 1 is the reference's rule.  (One pooled update per round -- what the
            // reference does per queue -- adapts K times slower: at C4, K = n = 200, the scale could not follow
            // the shrinking live set, chains froze and the live set collapsed onto clones.)
            const double facc = (double)ha / (double)(ha + hb);
            const double pw = (double)(K < s.nc ? K : s.nc);
            sc->scale *= exp(pw * (facc - s.facc) / (double)s.nc / s.facc);
        } else {                                             // tune_slice :1209-1239
            if (s_or & B2N_WARN_DOUBLING) sc->doubling = 1;
            const double ne = (double)(ha > 1 ? ha : 1), ncn = (double)hb;
            sc->scale *= fmin(fmax(ne * 2.0 / (ne + ncn), 0.5), 2.0);
            if (s_or & 0x80000000u) { sc->error = B2N_ERR_SLICE_FAIL; sc->done = 1; }
        }
        // ---- bound update due (sampler.py:648-651); first bound: enough calls AND efficiency below the
        //      threshold (sampler.py:407-409, 640-647)
        if (sc->phase == 0) {
            const double eff = 100.0 * (double)(s.it0 + sc->it) / (double)sc->ncall;
            if (sc->ncall >= s.first_min_ncall && eff < s.first_min_eff) sc->need_bound = 4;
        } else if (sc->ncall >= sc->ncall_last_update + s.update_interval) sc->need_bound = 1;
    }
}

// One launch between two chain launches: commit of the round whose chains have just finished, then the proposal
// of the next round (mode bit 0: commit, bit 1: propose).  R rounds = R + 1 of these instead of 2 R launches.
__global__ void __launch_bounds__(B2N_NS_THREADS, 1) ns_step_kernel(const NsDev s, int mode) {
    if (mode & 1) ns_commit_body(s);
    if (mode == 3) __syncthreads();       // the commit's global writes (live set, sorted order, scalars) are read below
    if (mode & 2) ns_propose_body(s);
}

// first nc columns of an (N, n) row-major block -> contiguous (N, nc)
__global__ void gather_cols_kernel(const double* __restrict__ src, int N, int n, int nc, double* __restrict__ dst) {
    const size_t tot = (size_t)N * nc;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (size_t)gridDim.x * blockDim.x) {
        const size_t r = e / nc, c = e - r * nc;
        dst[e] = src[r * n + c];
    }
}

__global__ void ns_clear_kernel(NsScalars* sc, B2nDyn* dyn, int bound_updated) {
    sc->need_bound = 0;
    if (bound_updated) { sc->ncall_last_update = sc->ncall; sc->phase = 1; }     // a bound exists from now on
    dyn->skip = 0;
}

// ---------------------------------------------------------------------------------------------
static int ns_alloc(b2n_ctx* ctx, b2n_ns* ns, void** p, size_t bytes) {
    B2N_CUDA(ctx, cudaMalloc(p, bytes ? bytes : 8));
    ns->allocs.push_back(*p);
    return B2N_OK;
}

static int ns_alloc_dead(b2n_ctx* ctx, b2n_ns* ns, long long cap) {
    // (re)allocate the dead-point arrays with room for `cap` rows, keeping the first `it` rows
    NsDev& d = ns->d;
    const size_t n = d.n;
    void* nu[5];
    const size_t bytes[5] = {(size_t)cap * n * 8, (size_t)cap * n * 8, (size_t)cap * 8, (size_t)cap * 8, (size_t)cap * 4};
    for (int i = 0; i < 5; i++) B2N_CUDA(ctx, cudaMalloc(&nu[i], bytes[i] ? bytes[i] : 8));
    if (ns->dead_alloc[0]) {
        NsScalars h;
        B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        B2N_CUDA(ctx, b2n_copy_sync(ctx, &h, d.sc, sizeof(h), cudaMemcpyDeviceToHost));
        const size_t rows = (size_t)std::min<long long>(h.it, ns->dead_cap);
        const size_t keep[5] = {rows * n * 8, rows * n * 8, rows * 8, rows * 8, rows * 4};
        for (int i = 0; i < 5; i++) {
            if (keep[i]) B2N_CUDA(ctx, b2n_copy_sync(ctx, nu[i], ns->dead_alloc[i], keep[i], cudaMemcpyDeviceToDevice));
            cudaFree(ns->dead_alloc[i]);
        }
    }
    for (int i = 0; i < 5; i++) ns->dead_alloc[i] = nu[i];
    d.dead_u = (double*)nu[0]; d.dead_v = (double*)nu[1]; d.dead_logl = (double*)nu[2];
    d.dead_logvol = (double*)nu[3]; d.dead_ncall = (int*)nu[4];
    ns->dead_cap = cap;
    d.dead_cap = cap;
    return B2N_OK;
}

void b2n_ns_release(b2n_ctx* ctx) {
    if (!ctx || !ctx->ns) return;
    if (ctx->ns->gexec) cudaGraphExecDestroy(ctx->ns->gexec);
    for (void* p : ctx->ns->allocs) cudaFree(p);
    for (void* p : ctx->ns->dead_alloc) if (p) cudaFree(p);
    delete ctx->ns;
    ctx->ns = nullptr;
}

// one chain-entry call in device-paced mode (plan_only: just report chains_per_cta)
static int ns_chain_call(b2n_ctx* ctx, b2n_ns* ns, bool plan_only) {
    NsDev& d = ns->d;
    b2n_chain_args a;
    memset(&a, 0, sizeof(a));
    a.nchain = d.K; a.ndim = d.n; a.ncdim = d.nc; a.model_id = ns->cfg.model_id;
    a.u0 = d.u0; a.ell = nullptr; a.dimflags = ns->has_flags ? ns->dimflags.data() : nullptr;
    a.seed = d.seed;
    const int mode = ctx->ptr_mode;
    ctx->ptr_mode = B2N_PTR_DEVICE;
    ctx->dyn.active = true;
    ctx->dyn.plan_only = plan_only;
    ctx->dyn.dev = d.dyn; ctx->dyn.order = d.order; ctx->dyn.cta = d.cta;
    ctx->dyn.max_cta = d.cpc > 0 ? d.K / d.cpc + d.Kell : 1;
    int st;
    if (ns->phase == 0) {
        if (plan_only) { ctx->dyn.cpc = 1; st = B2N_OK; }
        else st = b2n_unitcube_batch(ctx, &a, d.o_u, d.o_v, d.o_logl, d.o_ncall, d.o_flags);
    } else if (d.sampler == 3 && ns->friends) {
        st = b2n_friends_unif_dev(ctx, &a, d.N, ns->fr_kind, d.live_u, ns->fr_ctrs_t, ns->fr_axes, ns->fr_axinv, d.o_u,
                                  d.o_v, d.o_logl, d.o_ncall, d.o_i0, d.o_flags);
    } else if (d.sampler == 3) {
        if (plan_only) { ctx->dyn.cpc = 1; st = B2N_OK; }
        else st = b2n_unif_batch(ctx, &a, d.o_u, d.o_v, d.o_logl, d.o_ncall, d.o_i0, d.o_flags);
    } else if (d.sampler == 0)
        st = b2n_rwalk_batch(ctx, &a, ns->cfg.steps, d.o_u, d.o_v, d.o_logl, d.o_i0, d.o_i1, d.o_ncall);
    else if (d.sampler == 1)
        st = b2n_rslice_batch(ctx, &a, ns->cfg.steps, 0, d.o_u, d.o_v, d.o_logl, d.o_i0, d.o_i1, d.o_ncall, d.o_flags);
    else
        st = b2n_slice_batch(ctx, &a, ns->cfg.steps, 0, d.o_u, d.o_v, d.o_logl, d.o_i0, d.o_i1, d.o_ncall, d.o_flags);
    ctx->dyn.active = false;
    ctx->dyn.plan_only = false;
    ctx->ptr_mode = mode;
    return st;
}

#define B2N_NS_GRAPH_ROUNDS 16

// everything that is baked into the arguments of the kernels of a round
static unsigned long long ns_launch_key(b2n_ctx* ctx, b2n_ns* ns, size_t smem) {
    unsigned long long h = 1469598103934665603ULL;
    auto mix = [&](unsigned long long v) { h ^= v; h *= 1099511628211ULL; };
    const unsigned char* raw = reinterpret_cast<const unsigned char*>(&ns->d);      // NsDev is passed BY VALUE to the step
    for (size_t i = 0; i < sizeof(NsDev); i++) mix(raw[i]);                         // kernel (zero-initialised: no stray padding)
    mix((unsigned long long)ns->phase); mix((unsigned long long)(uintptr_t)ctx->b_axesT.p); mix((unsigned long long)smem);
    mix((unsigned long long)(uintptr_t)ctx->stream); mix((unsigned long long)ns->cfg.steps);
    mix((unsigned long long)ns->cfg.model_id); mix((unsigned long long)ctx->min_cpc); mix((unsigned long long)ctx->bK);
    return h ? h : 1;
}

static size_t ns_propose_smem(const NsDev& d) {
    return (size_t)(B2N_NS_THREADS / 32) * d.nc * 8 + (size_t)((d.Kell + 1) & ~1) * 8 + (size_t)d.K * 8 +
           (size_t)(d.Kell + 2) * 4 + 64;
}
static size_t ns_commit_smem(const NsDev& d) {
    const size_t NA = (size_t)(d.N - d.K);
    return (NA + (NA & 1)) * 8 + (size_t)d.Kpad * 8 + NA * 4 + (size_t)d.Kpad * 4 + 64;
}
static size_t ns_sort_smem(const NsDev& d) { return (size_t)d.Npad * 12 + 64; }

// A bound update is a chain of ~45 small dependent kernels with a dozen host round trips; with other replicas' chain
// CTAs filling every SM each of them used to wait its turn (68 updates cost 2.5 s per run at 48 replicas in flight
// against 0.18 s alone).  It runs on the context's HIGH-PRIORITY stream: its CTAs are placed before the pending CTAs
// of normal-priority grids.  The main stream is idle here (the rounds were synchronised).
struct StreamSwap {
    b2n_ctx* c; cudaStream_t keep; bool on;
    explicit StreamSwap(b2n_ctx* ctx) : c(ctx), keep(ctx->stream), on(ctx->own_stream && ctx->stream_hi != nullptr) {
        if (on) { cudaStreamSynchronize(keep); c->stream = c->stream_hi; }
    }
    ~StreamSwap() { if (on) { cudaStreamSynchronize(c->stream_hi); c->stream = keep; } }
};

// ---- friends mode --------------------------------------------------------------------------------------------------
static int ns_friends_alloc(b2n_ctx* ctx, b2n_ns* ns) {
    if (ns->fr_cov) return B2N_OK;            // (kept with the run's other allocations across runs of the same shape)
    const size_t n = ns->d.n, nn = n * n;
    B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->fr_cov, nn * 8));
    B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->fr_am, nn * 8));
    B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->fr_axes, nn * 8));
    B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->fr_axinv, nn * 8));
    B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->fr_ctrs_t, (size_t)ns->d.N * n * 8));
    return B2N_OK;
}

// the common axes as the one-"ellipsoid" resident bound the chain kernels read (get_random_axes returns self.axes,
// bounding.py:995-997 / 1262-1264).  The friends bounds have no ellipsoid centre: row 0 of the live set fills that slot, which no
// kernel of this mode reads (the uniform sampler of this mode draws around the live points themselves).
static int ns_friends_resident(b2n_ctx* ctx, b2n_ns* ns) {
    B2N_TRY(b2n_bound_set_dev(ctx, 1, ns->d.n, ns->d.live_u, ns->fr_am, ns->fr_axes, &ns->fr_logvol));
    ns->fr_serial = ctx->bound_serial;
    return B2N_OK;
}

// make the bound in fr_* the run's bound: resident axes, centres = the live set, ctrs_t = live_u @ axes_inv (all N rows)
static int ns_friends_adopt(b2n_ctx* ctx, b2n_ns* ns) {
    NsDev& d = ns->d;
    B2N_TRY(ns_friends_resident(ctx, ns));
    B2N_TRY(b2n_friends_transform_dev(ctx, d.live_u, d.N, d.n, ns->fr_axinv, ns->fr_ctrs_t));
    ns->friends = ns->fr_ready = true;
    return B2N_OK;
}

extern "C" {

int b2n_ns_create(b2n_ctx* ctx, const b2n_ns_config* c, int64_t dead_capacity) {
    if (!ctx || !c) return B2N_ERR_ARG;
    if (c->model_id < 0 || c->model_id >= (int)ctx->models.size()) return B2N_ERR_ARG;
    const int n = ctx->models[c->model_id].ndim;
    if (c->ndim != n || c->nlive < 2 || c->batch < 1 || c->batch >= c->nlive || c->steps < 1 || c->sampler < 0 ||
        c->sampler > 3 || c->ncdim < 1 || c->ncdim > n)
        return b2n_fail(ctx, B2N_ERR_ARG, "b2n_ns_create: need 1 <= batch < nlive, steps >= 1, sampler in {0,1,2,3}, ndim == model ndim");
    if ((c->sampler == 1 || c->sampler == 2) && c->ncdim != n) return b2n_fail(ctx, B2N_ERR_ARG, "slice samplers need ncdim == ndim");
    int Npad = 2;
    while (Npad < c->nlive) Npad <<= 1;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t want_cap = std::max<int64_t>(dead_capacity, (int64_t)c->batch);
    const bool reuse = ctx->ns && !ctx->ns->active && ctx->ns->d.N == c->nlive && ctx->ns->d.n == n &&
                       ctx->ns->d.nc == c->ncdim && ctx->ns->d.K == c->batch;
    if (!reuse) b2n_ns_release(ctx);
    b2n_ns* ns = reuse ? ctx->ns : new b2n_ns();
    ctx->ns = ns;
    ns->cfg = *c;
    ns->has_flags = false;
    if (c->dimflags) { ns->dimflags.assign(c->dimflags, c->dimflags + n); ns->has_flags = true; }
    ns->cfg.dimflags = nullptr;
    NsDev& d = ns->d;
    if (!reuse) memset(&d, 0, sizeof(d));
    d.N = c->nlive; d.n = n; d.nc = c->ncdim; d.K = c->batch; d.Kell = 1; d.strict = 1; d.sampler = c->sampler;
    d.Npad = Npad;
    d.Kpad = 2;
    while (d.Kpad < c->batch) d.Kpad <<= 1;
    // threads of the single-CTA step kernel (B2N_NS_THREADS=256|512 for experiments: no consistent effect measured,
    // profiles/r2*_scan*.jsonl)
    d.threads = B2N_NS_THREADS;
    if (const char* e = getenv("B2N_NS_THREADS")) d.threads = atoi(e) >= 1024 ? 1024 : (atoi(e) >= 512 ? 512 : 256);
    d.dlogz = c->dlogz; d.facc = c->facc; d.maxiter = c->maxiter; d.maxcall = c->maxcall;
    d.update_interval = c->update_interval; d.seed = c->seed; d.chain0 = c->chain0;
    d.first_min_ncall = c->first_min_ncall; d.first_min_eff = c->first_min_eff; d.it0 = c->it0;
    d.logl_max = c->use_logl_max ? c->logl_max : (double)INFINITY;
    ns->phase = c->unit_cube_phase ? 0 : 1;
    ns->bK = 0;
    ns->friends = ns->fr_ready = false;          // every run starts in ellipsoid mode
    d.friends = 0; d.fr_axes_inv = nullptr; d.fr_ctrs_t = nullptr;
    const size_t N = d.N, K = d.K;
    if (!reuse) {
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.live_u, N * n * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.live_v, N * n * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.live_logl, N * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.sc, sizeof(NsScalars)));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.dyn, sizeof(B2nDyn)));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.sidx, N * 4));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.skey, N * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.tidx, N * 4));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.tkey, N * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.u0, K * n * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.order, K * 4));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.cta, (K + N + 8) * sizeof(int3)));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.o_u, K * n * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.o_v, K * n * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.o_logl, K * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.o_i0, K * 4));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.o_i1, K * 4));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.o_ncall, K * 4));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&d.o_flags, K * 4));
        // device copy of the bound b2n_ns_update_bound builds (bounding.py:1493: a leaf has >= 2 ncdim points)
        const size_t nc = d.nc, nn = nc * nc;
        ns->Kmax = (int)std::max<size_t>(1, N / std::max<size_t>(2 * nc, 1));
        const size_t Km = ns->Kmax;
        B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->bd_ctrs, Km * nc * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->bd_covs, Km * nn * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->bd_ams, Km * nn * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->bd_axes, Km * nn * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->bd_axlens, Km * nc * 8));
        B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->bd_logvols, Km * 8));
        if (nc != (size_t)n) B2N_TRY(ns_alloc(ctx, ns, (void**)&ns->bd_points, N * nc * 8));
        B2N_TRY(ns_alloc_dead(ctx, ns, want_cap));
    } else if (ns->dead_cap < want_cap) {
        for (void*& pp : ns->dead_alloc) { if (pp) cudaFree(pp); pp = nullptr; }     // (nothing to keep from the last run)
        B2N_TRY(ns_alloc_dead(ctx, ns, want_cap));
    } else {
        d.dead_cap = want_cap;          // the capacity the caller asked for (the allocation may be larger)
    }
    cudaStream_t st = ctx->stream;      // stream-ordered clears (no device-wide synchronisation)
    B2N_CUDA(ctx, cudaMemsetAsync(d.o_i0, 0, K * 4, st));          // (the unit-cube sampler writes no counters)
    B2N_CUDA(ctx, cudaMemsetAsync(d.o_i1, 0, K * 4, st));          // (the uniform sampler writes no second counter)
    B2N_CUDA(ctx, cudaMemsetAsync(d.o_flags, 0, K * 4, st));
    B2N_CUDA(ctx, cudaMemsetAsync(d.sc, 0, sizeof(NsScalars), st));
    B2N_CUDA(ctx, cudaMemsetAsync(d.dyn, 0, sizeof(B2nDyn), st));
    ns->active = true;
    return B2N_OK;
}

int b2n_ns_destroy(b2n_ctx* ctx) {
    if (!ctx) return B2N_ERR_ARG;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->ns) ctx->ns->active = false;          // allocations are kept for the next run of the same shape
    return B2N_OK;
}

int b2n_ns_set_state(b2n_ctx* ctx, const double* live_u, const double* live_v, const double* live_logl,
                     double logvol, double logz, double loglstar, int64_t it, int64_t ncall, double scale) {
    if (!ctx || !ctx->ns || !ctx->ns->active || !live_u || !live_v || !live_logl) return B2N_ERR_ARG;
    b2n_ns* ns = ctx->ns;
    NsDev& d = ns->d;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t N = d.N, n = d.n;
    B2N_CUDA(ctx, b2n_copy_sync(ctx, d.live_u, live_u, N * n * 8, cudaMemcpyHostToDevice));
    B2N_CUDA(ctx, b2n_copy_sync(ctx, d.live_v, live_v, N * n * 8, cudaMemcpyHostToDevice));
    B2N_CUDA(ctx, b2n_copy_sync(ctx, d.live_logl, live_logl, N * 8, cudaMemcpyHostToDevice));
    NsScalars h;
    memset(&h, 0, sizeof(h));
    h.it = 0;                       // rows of the device dead buffer; the caller keeps its own offset
    (void)it;
    h.ncall = ncall; h.ncall_last_update = ncall;
    h.logvol = logvol; h.logz = logz; h.loglstar = loglstar; h.scale = scale;
    h.lmax = -1e300; h.delta_logz = 1e300;
    h.phase = ns->phase;
    B2N_CUDA(ctx, b2n_copy_sync(ctx, d.sc, &h, sizeof(h), cudaMemcpyHostToDevice));
    // (stream-ordered: a legacy-default-stream memset is NOT ordered against this context's non-blocking stream -- under
    //  load it landed between a proposal and its chain launch and zeroed the round's threshold: round 2, 32 replicas)
    B2N_CUDA(ctx, cudaMemsetAsync(d.dyn, 0, sizeof(B2nDyn), ctx->stream));
    const size_t smem = ns_sort_smem(d);
    if (smem > (size_t)ctx->max_smem_optin) return b2n_fail(ctx, B2N_ERR_UNSUPPORTED, "nlive too large for the one-CTA sort of b2n_ns");
    B2N_TRY(b2n_func_smem(ctx, (const void*)(ns_sort_kernel), (size_t)(smem)));
    ns_sort_kernel<<<1, B2N_NS_THREADS, smem, ctx->stream>>>(d);
    B2N_LAUNCH_CHECK(ctx);
    return B2N_OK;
}

static int ns_status(b2n_ctx* ctx, b2n_ns_status* out) {
    NsScalars* h = reinterpret_cast<NsScalars*>(ctx->pinned);
    B2N_CUDA(ctx, cudaMemcpyAsync(h, ctx->ns->d.sc, sizeof(NsScalars), cudaMemcpyDeviceToHost, ctx->stream));
    if (ctx->min_cpc > 1) {
        // a context that shares the GPU (b2n_set_chain_pack > 1: replicas) waits for its block of rounds -- milliseconds --
        // ASLEEP: dozens of host threads spinning in cudaStreamSynchronize starve the ones that have work to do
        if (!ctx->ev_block) B2N_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_block, cudaEventBlockingSync | cudaEventDisableTiming));
        B2N_CUDA(ctx, cudaEventRecord(ctx->ev_block, ctx->stream));
        B2N_CUDA(ctx, cudaEventSynchronize(ctx->ev_block));
    } else {
        B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (out) {
        out->it = h->it; out->ncall = h->ncall; out->rounds = h->round;
        out->logz = h->logz; out->logvol = h->logvol; out->loglstar = h->loglstar; out->lmax = h->lmax;
        out->delta_logz = h->delta_logz; out->scale = h->scale;
        out->done = h->done; out->need_bound = h->need_bound; out->doubling = h->doubling; out->error = h->error;
        out->ncall_last_update = h->ncall_last_update;
    }
    return B2N_OK;
}

int b2n_ns_status_get(b2n_ctx* ctx, b2n_ns_status* out) {
    if (!ctx || !ctx->ns || !ctx->ns->active || !out) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    return ns_status(ctx, out);
}

int b2n_ns_run(b2n_ctx* ctx, int32_t max_rounds, int32_t check_every, b2n_ns_status* out) {
    if (!ctx || !ctx->ns || !ctx->ns->active || max_rounds < 0) return B2N_ERR_ARG;
    b2n_ns* ns = ctx->ns;
    NsDev& d = ns->d;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    if (ctx->peer.total > 0) return b2n_fail(ctx, B2N_ERR_UNSUPPORTED, "b2n_ns_run: gather mode must be off");
    d.friends = 0; d.fr_axes_inv = nullptr; d.fr_ctrs_t = nullptr;
    if (ns->phase == 0) {            // unit-cube rounds: no bound yet
        d.Kell = 1;
        d.ctrs = d.ams = d.logvols = nullptr;
    } else if (ns->friends) {        // one common shape: the chains read its axes as the one resident "ellipsoid"
        if (!ns->fr_ready) return b2n_fail(ctx, B2N_ERR_ARG, "friends mode: no bound yet (b2n_ns_update_friends / b2n_ns_set_friends)");
        if (ctx->bound_serial != ns->fr_serial) B2N_TRY(ns_friends_resident(ctx, ns));   // someone replaced it since
        d.Kell = 1;
        d.ctrs = d.ams = d.logvols = nullptr;
        d.friends = 1;
        if (d.sampler == 3) { d.fr_axes_inv = ns->fr_axinv; d.fr_ctrs_t = ns->fr_ctrs_t; }
    } else {
        if (ctx->bK < 1 || ctx->bn != d.nc) return b2n_fail(ctx, B2N_ERR_ARG, "resident bound missing or of wrong dimension (b2n_bound_set)");
        if (!ctx->b_ctrs.p || !ctx->b_ams.p || !ctx->b_logvols.p || ctx->h_logvols.empty())
            return b2n_fail(ctx, B2N_ERR_ARG, "b2n_ns_run needs the full resident bound (ctrs, ams, logvols)");
        d.Kell = ctx->bK;
        d.ctrs = ctx->b_ctrs.as<double>(); d.ams = ctx->b_ams.as<double>(); d.logvols = ctx->b_logvols.as<double>();
    }
    d.strict = ns->cfg.strict_contains;
    if ((size_t)d.K / 1 + (size_t)d.Kell + 8 > (size_t)d.K + (size_t)d.N + 8)
        return b2n_fail(ctx, B2N_ERR_UNSUPPORTED, "too many ellipsoids for the round worklist");
    B2N_TRY(ns_chain_call(ctx, ns, true));               // chains per CTA the chain kernel plans for
    d.cpc = ctx->dyn.cpc;
    const size_t smem = std::max(ns_propose_smem(d), ns_commit_smem(d));
    if (smem + 2048 > (size_t)ctx->max_smem_optin)
        return b2n_fail(ctx, B2N_ERR_UNSUPPORTED, "nlive / batch too large for the one-CTA kernels of b2n_ns_run");
    B2N_TRY(b2n_func_smem(ctx, (const void*)(ns_step_kernel), (size_t)(smem)));
    if (check_every < 1) check_every = max_rounds > 0 ? max_rounds : 1;
    int left = max_rounds;
    b2n_ns_status st;
    memset(&st, 0, sizeof(st));
    // graphs: chain samplers without per-dimension flags (their entry points then issue no copies), timing off
    // OPT-IN (B2N_NS_GRAPH=1): measured on B200 (profiles/r2c_replica_scan.jsonl vs r2c_nograph.log) the replay is not
    // faster than the plain launches -- one run alone 12.9e6 vs 13.9e6 calls/s, 16 replicas in flight 4.7e7 vs 6.5e7 --
    // the rounds are bound by the dependent kernels' execution latency on the device, not by the host's launch rate.
    const char* genv = getenv("B2N_NS_GRAPH");
    const bool graph_ok = (genv && genv[0] == '1') && !ns->has_flags && !ctx->timing && (ns->phase == 0 || d.sampler != 3);
    const unsigned long long key = ns_launch_key(ctx, ns, smem);
    while (left > 0) {
        const int chunk = std::min(left, (int)check_every);
        // R rounds = R x ( commit of the pending round + proposal of the next | chains ) + one closing commit
        int r = 0;
        if (graph_ok && ns->warm_key == key && chunk >= B2N_NS_GRAPH_ROUNDS) {
            if (!ns->gexec || ns->gkey != key) {
                if (ns->gexec) { cudaGraphExecDestroy(ns->gexec); ns->gexec = nullptr; }
                cudaGraph_t g = nullptr;
                B2N_CUDA(ctx, cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
                int cst = B2N_OK;
                for (int q = 0; q < B2N_NS_GRAPH_ROUNDS && cst == B2N_OK; q++) {
                    ns_step_kernel<<<1, d.threads, smem, ctx->stream>>>(d, 3);
                    cst = ns_chain_call(ctx, ns, false);
                }
                const cudaError_t ce = cudaStreamEndCapture(ctx->stream, &g);
                if (cst != B2N_OK || ce != cudaSuccess || !g) {
                    if (g) cudaGraphDestroy(g);
                    cudaGetLastError();
                    return cst != B2N_OK ? cst : b2n_fail(ctx, B2N_ERR_CUDA, "stream capture of the round graph failed");
                }
                const cudaError_t ie = cudaGraphInstantiate(&ns->gexec, g, 0);
                cudaGraphDestroy(g);
                if (ie != cudaSuccess) { ns->gexec = nullptr; cudaGetLastError(); return b2n_fail(ctx, B2N_ERR_CUDA, "cudaGraphInstantiate failed"); }
                ns->gkey = key;
            }
            for (; r + B2N_NS_GRAPH_ROUNDS <= chunk; r += B2N_NS_GRAPH_ROUNDS) {
                B2N_CUDA(ctx, cudaGraphLaunch(ns->gexec, ctx->stream));
                ctx->launches += 2 * B2N_NS_GRAPH_ROUNDS;
            }
        }
        for (; r < chunk; r++) {
            ns_step_kernel<<<1, d.threads, smem, ctx->stream>>>(d, 3);
            B2N_LAUNCH_CHECK(ctx);
            B2N_TRY(ns_chain_call(ctx, ns, false));
        }
        ns->warm_key = key;             // these very launches have been issued once outside a capture (buffers exist)
        ns_step_kernel<<<1, d.threads, smem, ctx->stream>>>(d, 1);
        B2N_LAUNCH_CHECK(ctx);
        left -= chunk;
        B2N_TRY(ns_status(ctx, &st));
        if (st.done || st.need_bound) break;
    }
    if (max_rounds == 0) B2N_TRY(ns_status(ctx, &st));
    if (out) *out = st;
    if (st.error) {
        snprintf(ctx->err, sizeof(ctx->err), "device rounds stopped with status %d after round %lld (phase %d, sampler %d, it %lld, ncall %lld)",
                 st.error, (long long)st.rounds, ns->phase, d.sampler, (long long)st.it, (long long)st.ncall);
        return st.error;
    }
    return B2N_OK;
}

__global__ void ns_set_counters_kernel(NsScalars* sc, long long rounds, long long ncall_last_update, int doubling) {
    sc->round = rounds;
    sc->ncall_last_update = ncall_last_update;
    sc->doubling = doubling;
}

int b2n_ns_set_counters(b2n_ctx* ctx, int64_t rounds, int64_t ncall_last_update, int32_t doubling) {
    if (!ctx || !ctx->ns || !ctx->ns->active || rounds < 0) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    ns_set_counters_kernel<<<1, 1, 0, ctx->stream>>>(ctx->ns->d.sc, rounds, ncall_last_update, doubling);
    B2N_LAUNCH_CHECK(ctx);
    return B2N_OK;
}

int b2n_ns_bound_updated(b2n_ctx* ctx) {
    if (!ctx || !ctx->ns || !ctx->ns->active) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    ns_clear_kernel<<<1, 1, 0, ctx->stream>>>(ctx->ns->d.sc, ctx->ns->d.dyn, 1);
    B2N_LAUNCH_CHECK(ctx);
    ctx->ns->phase = 1;              // the unit-cube phase ends with the first bound (sampler.py:640-647)
    return B2N_OK;
}

int b2n_ns_update_bound(b2n_ctx* ctx, int32_t multi, double enlarge, int32_t* nells, double* logvol, uint32_t* warn) {
    if (!ctx || !ctx->ns || !ctx->ns->active || !(enlarge > 0.0)) return B2N_ERR_ARG;
    b2n_ns* ns = ctx->ns;
    NsDev& d = ns->d;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    if (ns->friends) return b2n_fail(ctx, B2N_ERR_ARG, "b2n_ns_update_bound: this run holds a friends bound (b2n_ns_update_friends)");
    StreamSwap swap_(ctx);
    const int n = d.n, nc = d.nc, N = d.N;
    const double* pts = d.live_u;
    if (nc != n) {                  // the bound lives in the first ncdim coordinates (sampler.py:497)
        gather_cols_kernel<<<(unsigned)std::min<size_t>(((size_t)N * nc + 255) / 256, 1024), 256, 0, ctx->stream>>>(
            d.live_u, N, n, nc, ns->bd_points);
        B2N_LAUNCH_CHECK(ctx);
        pts = ns->bd_points;
    }
    const int mode = ctx->ptr_mode;
    ctx->ptr_mode = B2N_PTR_DEVICE;          // points and outputs are device arrays of this run
    int32_t K = 1;
    uint32_t w = 0;
    int st;
    if (multi)
        st = b2n_multi_decompose(ctx, pts, N, nc, ns->Kmax, &K, nullptr, ns->bd_ctrs, ns->bd_covs, ns->bd_ams, ns->bd_axes,
                                 ns->bd_axlens, ns->bd_logvols, &w);
    else
        st = b2n_bounding_ellipsoid(ctx, pts, N, nc, ns->bd_ctrs, ns->bd_covs, ns->bd_ams, ns->bd_axes, ns->bd_axlens,
                                    ns->bd_logvols, &w);
    ctx->ptr_mode = mode;
    if (st != B2N_OK) return st;
    std::vector<double> lv(K);
    B2N_CUDA(ctx, cudaMemcpyAsync(lv.data(), ns->bd_logvols, (size_t)K * 8, cudaMemcpyDeviceToHost, ctx->stream));
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (enlarge != 1.0) {
        // sampler.py:506-508 -> scalar branch of MultiEllipsoid.scale_to_logvol (bounding.py:487-489): every
        // ellipsoid is shifted by the same ln(enlarge)
        // (the targets are formed with the host classes' arithmetic, so that this entry and the host route --
        //  B200MultiEllipsoid.scale_to_logvol(logvol + ln enlarge) -- are bit-identical: (L + x) - L != x)
        std::vector<double> tg(K);
        if (multi) {
            double hi = -INFINITY, se = 0.0;
            for (double x : lv) hi = std::max(hi, x);
            for (double x : lv) se += exp(x - hi);
            const double L = hi + log(se), T = L + log(enlarge);
            for (int k = 0; k < K; k++) tg[k] = lv[k] + (T - L);
        } else {
            tg[0] = lv[0] + log(enlarge);
        }
        ctx->ptr_mode = B2N_PTR_DEVICE;
        st = b2n_scale_to_logvol(ctx, K, nc, ns->bd_covs, ns->bd_ams, ns->bd_axes, ns->bd_axlens, ns->bd_logvols, tg.data());
        ctx->ptr_mode = mode;
        if (st != B2N_OK) return st;
        B2N_CUDA(ctx, cudaMemcpyAsync(lv.data(), ns->bd_logvols, (size_t)K * 8, cudaMemcpyDeviceToHost, ctx->stream));
        B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    B2N_TRY(b2n_bound_set_dev(ctx, K, nc, ns->bd_ctrs, ns->bd_ams, ns->bd_axes, lv.data()));
    ns->bK = K;
    ns->bd_hlogvols = lv;
    if (nells) *nells = K;
    if (logvol) {
        double hi = -INFINITY, se = 0.0;
        for (double x : lv) hi = std::max(hi, x);
        for (double x : lv) se += exp(x - hi);
        *logvol = hi + log(se);
    }
    if (warn) *warn = w;
    return B2N_OK;
}

int b2n_ns_get_bound(b2n_ctx* ctx, int32_t max_ells, double* ctrs, double* covs, double* ams, double* axes,
                     double* axlens, double* logvols) {
    if (!ctx || !ctx->ns || !ctx->ns->active) return B2N_ERR_ARG;
    b2n_ns* ns = ctx->ns;
    if (ns->bK < 1 || max_ells < ns->bK) return b2n_fail(ctx, B2N_ERR_ARG, "b2n_ns_get_bound: no device-built bound / max_ells too small");
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t K = ns->bK, nc = ns->d.nc, nn = nc * nc;
    if (ctrs) B2N_CUDA(ctx, b2n_copy_sync(ctx, ctrs, ns->bd_ctrs, K * nc * 8, cudaMemcpyDeviceToHost));
    if (covs) B2N_CUDA(ctx, b2n_copy_sync(ctx, covs, ns->bd_covs, K * nn * 8, cudaMemcpyDeviceToHost));
    if (ams) B2N_CUDA(ctx, b2n_copy_sync(ctx, ams, ns->bd_ams, K * nn * 8, cudaMemcpyDeviceToHost));
    if (axes) B2N_CUDA(ctx, b2n_copy_sync(ctx, axes, ns->bd_axes, K * nn * 8, cudaMemcpyDeviceToHost));
    if (axlens) B2N_CUDA(ctx, b2n_copy_sync(ctx, axlens, ns->bd_axlens, K * nc * 8, cudaMemcpyDeviceToHost));
    if (logvols) memcpy(logvols, ns->bd_hlogvols.data(), K * 8);
    return B2N_OK;
}

int b2n_ns_update_friends(b2n_ctx* ctx, int32_t kind, double enlarge, int32_t nboot, int32_t use_clustering,
                          double* logvol, double* radius, int32_t* nclusters) {
    if (!ctx || !ctx->ns || !ctx->ns->active || (kind != 0 && kind != 1) || !(enlarge > 0.0) || nboot < 0) return B2N_ERR_ARG;
    if (nboot > B2N_NS_FRIENDS_MAX_BOOT) return b2n_fail(ctx, B2N_ERR_ARG, "b2n_ns_update_friends: nboot <= 255 (bootstrap chain ids)");
    b2n_ns* ns = ctx->ns;
    NsDev& d = ns->d;
    if (d.nc != d.n) return b2n_fail(ctx, B2N_ERR_ARG, "the friends bounds need ncdim == ndim");
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    B2N_TRY(ns_friends_alloc(ctx, ns));
    StreamSwap swap_(ctx);
    const int n = d.n, N = d.N;
    const size_t nn = (size_t)n * n;
    NsScalars h;                                 // round index: the bootstrap streams of this update
    B2N_CUDA(ctx, b2n_copy_sync(ctx, &h, d.sc, sizeof(h), cudaMemcpyDeviceToHost));
    if (!ns->fr_ready) {                         // no previous metric: the identity, RadFriends(ndim)'s (bounding.py:749-762)
        std::vector<double> eye(nn, 0.0);
        for (int i = 0; i < n; i++) eye[(size_t)i * n + i] = 1.0;
        B2N_CUDA(ctx, b2n_copy_sync(ctx, ns->fr_am, eye.data(), nn * 8, cudaMemcpyHostToDevice));
    }
    const int mode = ctx->ptr_mode;
    ctx->ptr_mode = B2N_PTR_DEVICE;              // the live set and the outputs are device arrays of this run
    double lv = 0.0, r = 0.0;
    int32_t ncl = 1;
    // am_prev = the run's current am, overwritten in place by the new one (read by the first kernel of the update,
    // written by its last copy, in stream order)
    const int st = b2n_friends_update(ctx, d.live_u, N, n, kind, use_clustering, ns->fr_am, nboot, d.seed,
                                      B2N_NS_FRIENDS_BOOT_CHAIN + ((unsigned long long)h.round << 8), ns->fr_cov, ns->fr_am,
                                      ns->fr_axes, ns->fr_axinv, &lv, &r, &ncl);
    ctx->ptr_mode = mode;
    if (st != B2N_OK) return st;
    if (enlarge != 1.0) {
        // sampler.py:506-508: scale_to_logvol(logvol + ln enlarge), with the host class's arithmetic
        // (f = exp(((L + ln e) - L) / n), not e^(1/n): (L + x) - L != x) so that both routes are bit-identical
        const double T = lv + log(enlarge);
        const double f = exp((T - lv) / (double)n);
        B2N_TRY(b2n_friends_rescale_dev(ctx, n, ns->fr_cov, ns->fr_am, ns->fr_axes, ns->fr_axinv, f));
        lv = T;
    }
    ns->fr_kind = kind;
    ns->fr_logvol = lv;
    ns->fr_radius = r;
    ns->fr_ncl = ncl;
    B2N_TRY(ns_friends_adopt(ctx, ns));
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (logvol) *logvol = lv;
    if (radius) *radius = r;
    if (nclusters) *nclusters = ncl;
    return B2N_OK;
}

int b2n_ns_set_friends(b2n_ctx* ctx, int32_t kind, const double* cov, const double* am, const double* axes,
                       const double* axes_inv, double logvol) {
    if (!ctx || !ctx->ns || !ctx->ns->active || (kind != 0 && kind != 1) || !cov || !am || !axes || !axes_inv)
        return B2N_ERR_ARG;
    b2n_ns* ns = ctx->ns;
    if (ns->d.nc != ns->d.n) return b2n_fail(ctx, B2N_ERR_ARG, "the friends bounds need ncdim == ndim");
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    B2N_TRY(ns_friends_alloc(ctx, ns));
    const size_t nn = (size_t)ns->d.n * ns->d.n * 8;
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));          // (enqueued rounds may still read the previous bound)
    B2N_CUDA(ctx, b2n_copy_sync(ctx, ns->fr_cov, cov, nn, cudaMemcpyHostToDevice));
    B2N_CUDA(ctx, b2n_copy_sync(ctx, ns->fr_am, am, nn, cudaMemcpyHostToDevice));
    B2N_CUDA(ctx, b2n_copy_sync(ctx, ns->fr_axes, axes, nn, cudaMemcpyHostToDevice));
    B2N_CUDA(ctx, b2n_copy_sync(ctx, ns->fr_axinv, axes_inv, nn, cudaMemcpyHostToDevice));
    ns->fr_kind = kind;
    ns->fr_logvol = logvol;
    ns->fr_radius = NAN;                         // not known for an adopted bound
    ns->fr_ncl = 0;
    B2N_TRY(ns_friends_adopt(ctx, ns));
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return B2N_OK;
}

int b2n_ns_get_friends(b2n_ctx* ctx, double* cov, double* am, double* axes, double* axes_inv, double* logvol,
                       double* radius, int32_t* nclusters) {
    if (!ctx || !ctx->ns || !ctx->ns->active) return B2N_ERR_ARG;
    b2n_ns* ns = ctx->ns;
    if (!ns->fr_ready) return b2n_fail(ctx, B2N_ERR_ARG, "b2n_ns_get_friends: the run holds no friends bound");
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t nn = (size_t)ns->d.n * ns->d.n * 8;
    if (cov) B2N_CUDA(ctx, b2n_copy_sync(ctx, cov, ns->fr_cov, nn, cudaMemcpyDeviceToHost));
    if (am) B2N_CUDA(ctx, b2n_copy_sync(ctx, am, ns->fr_am, nn, cudaMemcpyDeviceToHost));
    if (axes) B2N_CUDA(ctx, b2n_copy_sync(ctx, axes, ns->fr_axes, nn, cudaMemcpyDeviceToHost));
    if (axes_inv) B2N_CUDA(ctx, b2n_copy_sync(ctx, axes_inv, ns->fr_axinv, nn, cudaMemcpyDeviceToHost));
    if (logvol) *logvol = ns->fr_logvol;
    if (radius) *radius = ns->fr_radius;
    if (nclusters) *nclusters = ns->fr_ncl;
    return B2N_OK;
}

int b2n_ns_reserve_dead(b2n_ctx* ctx, int64_t capacity) {
    if (!ctx || !ctx->ns || !ctx->ns->active) return B2N_ERR_ARG;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    if (capacity > ctx->ns->dead_cap) B2N_TRY(ns_alloc_dead(ctx, ctx->ns, capacity));
    else if (capacity > ctx->ns->d.dead_cap) ctx->ns->d.dead_cap = capacity;          // allocation already large enough
    ns_clear_kernel<<<1, 1, 0, ctx->stream>>>(ctx->ns->d.sc, ctx->ns->d.dyn, 0);   // clears need_bound == 3
    B2N_LAUNCH_CHECK(ctx);
    return B2N_OK;
}

int b2n_ns_get_live(b2n_ctx* ctx, double* live_u, double* live_v, double* live_logl) {
    if (!ctx || !ctx->ns || !ctx->ns->active) return B2N_ERR_ARG;
    NsDev& d = ctx->ns->d;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t N = d.N, n = d.n;
    if (live_u) B2N_CUDA(ctx, b2n_copy_sync(ctx, live_u, d.live_u, N * n * 8, cudaMemcpyDeviceToHost));
    if (live_v) B2N_CUDA(ctx, b2n_copy_sync(ctx, live_v, d.live_v, N * n * 8, cudaMemcpyDeviceToHost));
    if (live_logl) B2N_CUDA(ctx, b2n_copy_sync(ctx, live_logl, d.live_logl, N * 8, cudaMemcpyDeviceToHost));
    return B2N_OK;
}

int b2n_ns_get_dead(b2n_ctx* ctx, int64_t first, int64_t count, double* u, double* v, double* logl,
                    double* logvol, int32_t* ncall) {
    if (!ctx || !ctx->ns || first < 0 || count < 0) return B2N_ERR_ARG;
    NsDev& d = ctx->ns->d;
    B2N_CUDA(ctx, cudaSetDevice(ctx->device));
    B2N_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (first + count > ctx->ns->dead_cap) return B2N_ERR_ARG;
    const size_t n = d.n, f = (size_t)first, c = (size_t)count;
    if (c == 0) return B2N_OK;
    if (u) B2N_CUDA(ctx, b2n_copy_sync(ctx, u, d.dead_u + f * n, c * n * 8, cudaMemcpyDeviceToHost));
    if (v) B2N_CUDA(ctx, b2n_copy_sync(ctx, v, d.dead_v + f * n, c * n * 8, cudaMemcpyDeviceToHost));
    if (logl) B2N_CUDA(ctx, b2n_copy_sync(ctx, logl, d.dead_logl + f, c * 8, cudaMemcpyDeviceToHost));
    if (logvol) B2N_CUDA(ctx, b2n_copy_sync(ctx, logvol, d.dead_logvol + f, c * 8, cudaMemcpyDeviceToHost));
    if (ncall) B2N_CUDA(ctx, b2n_copy_sync(ctx, ncall, d.dead_ncall + f, c * 4, cudaMemcpyDeviceToHost));
    return B2N_OK;
}

}  // extern "C"
