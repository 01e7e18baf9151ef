// Exact surface-distance metrics of pairs of 2-D binary maps (tl_surface_distances): the Hausdorff distance, a
// percentile Hausdorff distance, the average symmetric surface distance and the normalized surface Dice.  The surface
// of a mask M is S(M) = M & ~binary_erosion(M) (cross structure, outside = 0): its nonzero pixels with a zero or an
// outside 4-neighbour.
//
// edt_row_kernel<SurfSrc, 1>  (edt_kernel.cuh) once per mask: h, the horizontal distance of every pixel to the
//                             nearest surface pixel in its row
// surface_col_kernel<M>       one CTA per map, one thread per column: the lower envelopes of both surfaces (EdtEnv),
//                             walked together (EdtWalk).  At a pixel of S(pred) the walk of S(target) gives s, the
//                             exact squared distance to S(target), and the other way round.  Per map: counts, the
//                             largest s, the fp64 sum of sqrt(s) and the count within the tolerance, reduced in a fixed
//                             order; the Hausdorff distance, ASSD and NSD; and every pixel's s as a key for the select
// surface_select_kernel<M>    one CTA per map: numpy's linear percentile of each direction from
//                             the exact (lo + 1)-th and (lo + 2)-th smallest keys (block_radix_select)
//
// Every distance is sqrt(float64(s)) of an integer s < 2^25, so the only roundings are the roots, the fp64 reductions
// and the final fp32 conversion.
//
// With a spacing per map (a non-null spacing, DESIGN §3.10) the column pass walks the weighted envelopes (EdtSpacing)
// and stores each surface pixel's packed offset (edt_pack) as its key; s is the fp64 value recomputed from it, the
// maxima are taken over the bits of s (monotone as uint64 for s >= 0) and the select runs over 64-bit keys.
#pragma once
#include <type_traits>
#include "edt_kernel.cuh"

namespace tl {

constexpr uint32_t kSurfNone = kEdtNone;  // key of a pixel off the surface: above every s (Metric::key)
constexpr int kSurfSelThreads = 512;

// floor(x / d) for x < 2^53: a reciprocal estimate, off by at most one, then corrected exactly in integers.  The
// 64-bit integer division it replaces is a call that spills in edt_row_kernel.
__device__ __forceinline__ size_t surf_div(size_t x, int d) {
    size_t q = (size_t)((double)x * __drcp_rn((double)d));
    if (q * d > x) --q;
    else if ((q + 1) * d <= x) ++q;
    return q;
}

// false exactly on the pixels of S(M) (the label of edt_row_kernel<SurfSrc, 1>); i is the flat index into [n][H][W]
struct SurfSrc {
    const uint8_t* m;
    int H, W;
    __device__ __forceinline__ bool operator()(size_t i) const {
        if (__ldg(m + i) == 0) return true;
        const size_t r = surf_div(i, W);
        const int c = (int)(i - r * W), u = (int)(r - surf_div(r, H) * H);
        return u > 0 && u < H - 1 && c > 0 && c < W - 1 && __ldg(m + i - W) != 0 && __ldg(m + i + W) != 0 &&
               __ldg(m + i - 1) != 0 && __ldg(m + i + 1) != 0;
    }
};

struct SurfArgs {
    uint32_t* h;        // [2][n][H][W]: the row pass of S(pred), then of S(target); overwritten by the envelopes
    uint32_t* keys;     // [2][n][H][W]: the walk value (s, or the packed offset) from each pixel of S(pred) to
                        // S(target), then from S(target) to S(pred); kSurfNone off the surface
    uint32_t* stats;    // [4][n]: |S(pred)|, |S(target)|, largest s of each direction (EdtUnit only); counts 0 on a
                        // map with an empty surface, whose outputs the column pass writes in full
    int n_maps, H, W;
    double tol;         // NSD tolerance
    double qq;          // percentile / 100
    float* out;         // [4][n]: hausdorff, hausdorff_percentile, assd, nsd
    const double* spacing;  // EdtSpacing: [n][2] (sy, sx) per map
};

// warp maxima and minima of 32- and 64-bit keys
__device__ __forceinline__ uint32_t surf_warp_max(uint32_t m) { return __reduce_max_sync(0xFFFFFFFFu, m); }
__device__ __forceinline__ uint32_t surf_warp_min(uint32_t m) { return __reduce_min_sync(0xFFFFFFFFu, m); }
__device__ __forceinline__ unsigned long long surf_warp_max(unsigned long long m) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    return m;
}
__device__ __forceinline__ unsigned long long surf_warp_min(unsigned long long m) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    return m;
}

// Metric: EdtUnit, or EdtSpacing of each map's spacing.  The maxima are taken over the keys (Metric::Key).
template <class Metric>
__global__ void __launch_bounds__(kEdtColThreads) surface_col_kernel(SurfArgs A) {
    using Key = typename Metric::Key;
    __shared__ double s_red[32];
    __shared__ Key s_max[2];
    __shared__ int s_has;  // bit 0: S(pred) is nonempty, bit 1: S(target) is
    const int H = A.H, W = A.W, n = A.n_maps;
    const size_t N = (size_t)H * W, nN = (size_t)n * N;
    for (int map = blockIdx.x; map < n; map += gridDim.x) {
        if (threadIdx.x == 0) s_max[0] = s_max[1] = 0u;
        uint32_t cnt[2] = {0u, 0u}, ntol = 0u;
        Key mx[2] = {0u, 0u};
        double sum = 0.0;
        const Metric m = Metric::of(A.spacing, map);
        for (int j = threadIdx.x; j < W; j += blockDim.x) {
            EdtEnv<Metric> env[2];
#pragma unroll
            for (int L = 0; L < 2; ++L) {
                env[L].col = A.h + L * nN + (size_t)map * N + j;
                env[L].stride = (size_t)W;
                env[L].top = -1;
                env[L].m = m;
            }
            for (int i = 0; i < H; ++i) {
#pragma unroll
                for (int L = 0; L < 2; ++L) {
                    const uint32_t hi = env[L].col[(size_t)i * W];
                    if (hi != kEdtNone) env[L].push(i, (int)hi, H);
                }
            }
            // a surface with a pixel has one in some row, and then every column's envelope holds that row: the
            // emptiness of either envelope is the same in every column
            const int has = (env[0].top >= 0 ? 1 : 0) | (env[1].top >= 0 ? 2 : 0);
            if (j == 0) s_has = has;
            if (has != 3) continue;
            EdtWalk<Metric> walk[2];
#pragma unroll
            for (int L = 0; L < 2; ++L) walk[L].start(env[L], H);
            uint32_t* kp = A.keys + (size_t)map * N + j;
            uint32_t* kt = kp + nN;
            for (int u = 0; u < H; ++u) {
                // walk values of pixel (u, j) towards S(pred) and S(target): 0 exactly on that surface
                const uint32_t sp = (uint32_t)walk[0].at(env[0], u), st = (uint32_t)walk[1].at(env[1], u);
                uint32_t k0 = kSurfNone, k1 = kSurfNone;
                if (sp == 0u) {
                    const double d = sqrt(m.sq(st));
                    k0 = st; ++cnt[0]; mx[0] = max(mx[0], m.key(st)); sum += d; ntol += d <= A.tol ? 1u : 0u;
                }
                if (st == 0u) {
                    const double d = sqrt(m.sq(sp));
                    k1 = sp; ++cnt[1]; mx[1] = max(mx[1], m.key(sp)); sum += d; ntol += d <= A.tol ? 1u : 0u;
                }
                kp[(size_t)u * W] = k0;
                kt[(size_t)u * W] = k1;
            }
        }
        // counts are below 2^25: exact in fp64
        const double np = block_sum((double)cnt[0], s_red), nt = block_sum((double)cnt[1], s_red);
        const double ntl = block_sum((double)ntol, s_red), total = block_sum(sum, s_red);
#pragma unroll
        for (int L = 0; L < 2; ++L) {
            const Key w = surf_warp_max(mx[L]);
            if ((threadIdx.x & 31) == 0) atomicMax(&s_max[L], w);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const int has = s_has;
            const float nan = __int_as_float(0x7FC00000), inf = __int_as_float(0x7F800000);
            float hd, assd, nsd;
            if (has == 3) {
                hd = (float)sqrt(m.key_sq(max(s_max[0], s_max[1])));
                assd = (float)(total / (np + nt));
                nsd = (float)(ntl / (np + nt));
            } else {  // one empty surface: infinitely far, nothing within the tolerance; both empty: undefined
                hd = assd = has ? inf : nan;
                nsd = has ? 0.f : nan;
                A.out[n + map] = hd;
            }
            A.out[map] = hd;
            A.out[2 * n + map] = assd;
            A.out[3 * n + map] = nsd;
            A.stats[map] = has == 3 ? (uint32_t)np : 0u;
            A.stats[n + map] = has == 3 ? (uint32_t)nt : 0u;
            if constexpr (std::is_same_v<Metric, EdtUnit>) {
                A.stats[2 * n + map] = s_max[0];
                A.stats[3 * n + map] = s_max[1];
            }
        }
        __syncthreads();  // s_red, s_max and s_has are reused by the next map
    }
}

// numpy's linear percentile (np.percentile's default) of the cnt distances sqrt(s) of one map and direction: the
// stored walk values below kSurfNone, ordered by Metric::key (the sentinel maps to the largest key, above every s).
// h >= cnt - 1 selects the largest s (rank cnt); EdtUnit reads it from *mx, its stored largest s, instead.  The
// interpolation is written without FMA contraction, as numpy evaluates it.
template <class Metric>
__device__ __forceinline__ double surface_percentile(const uint32_t* key, int N, uint32_t cnt, const uint32_t* mx,
                                                     double qq, const Metric& m, uint32_t* s_hist, uint32_t* s_digit,
                                                     uint32_t* s_k, typename Metric::Key* s_min) {
    using Key = typename Metric::Key;
    const double h = __dmul_rn((double)(cnt - 1u), qq);
    const bool last = h >= (double)(cnt - 1u);
    if constexpr (std::is_same_v<Metric, EdtUnit>) {
        if (last) return sqrt((double)*mx);
    }
    const double lo = last ? (double)(cnt - 1u) : floor(h), g = __dsub_rn(h, lo);
    // d[lo] is the (lo + 1)-th smallest s: the (lo + 1)-th largest ~key
    const RadixPickT<Key> pick = block_radix_select<kSurfSelThreads, Key>(
        [&](int i) { return ~m.key(__ldg(key + i)); }, N, (uint32_t)lo + 1u, s_hist, s_digit, s_k);
    const Key sa = ~pick.value;
    const double a = sqrt(m.key_sq(sa));
    if (last) return a;
    Key sb = sa;
    if (pick.k >= pick.count) {  // d[lo] ends its run of equal keys: d[lo + 1] is the smallest key above it
        if (threadIdx.x == 0) *s_min = ~(Key)0u;
        __syncthreads();
        Key v = ~(Key)0u;
        for (int i = threadIdx.x; i < N; i += kSurfSelThreads) {
            const Key k = m.key(__ldg(key + i));
            if (k > sa) v = min(v, k);
        }
        v = surf_warp_min(v);
        if ((threadIdx.x & 31) == 0) atomicMin(s_min, v);
        __syncthreads();
        sb = *s_min;
        __syncthreads();  // s_min is rewritten by the next call
    }
    const double b = sqrt(m.key_sq(sb)), diff = __dsub_rn(b, a);
    return g >= 0.5 ? __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, g))) : __dadd_rn(a, __dmul_rn(diff, g));
}

template <class Metric>
__global__ void __launch_bounds__(kSurfSelThreads) surface_select_kernel(SurfArgs A) {
    __shared__ uint32_t s_hist[256];
    __shared__ uint32_t s_digit, s_k;
    __shared__ typename Metric::Key s_min;
    const int n = A.n_maps, N = A.H * A.W;
    const size_t nN = (size_t)n * N;
    for (int map = blockIdx.x; map < n; map += gridDim.x) {
        const uint32_t np = A.stats[map], nt = A.stats[n + map];
        if (np == 0u) continue;  // an empty surface: the column pass wrote this map's outputs (uniform)
        const uint32_t* kp = A.keys + (size_t)map * N;
        const Metric m = Metric::of(A.spacing, map);
        const double pp = surface_percentile(kp, N, np, A.stats + 2 * n + map, A.qq, m, s_hist, &s_digit, &s_k, &s_min);
        const double pt = surface_percentile(kp + nN, N, nt, A.stats + 3 * n + map, A.qq, m, s_hist, &s_digit, &s_k, &s_min);
        if (threadIdx.x == 0) A.out[n + map] = (float)fmax(pp, pt);
    }
}

}  // namespace tl
