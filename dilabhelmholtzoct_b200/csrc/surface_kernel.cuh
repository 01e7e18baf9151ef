// Exact surface-distance metrics of pairs of 2-D binary maps (tl_surface_distances): the Hausdorff distance, a
// percentile Hausdorff distance, the average symmetric surface distance and the normalized surface Dice.  The surface
// of a mask M is S(M) = M & ~binary_erosion(M) (cross structure, outside = 0): its nonzero pixels with a zero or an
// outside 4-neighbour.
//
// edt_row_kernel<SurfSrc, 1>  (edt_kernel.cuh) once per mask: h, the horizontal distance of every pixel to the
//                             nearest surface pixel in its row
// surface_col_kernel          one CTA per map, one thread per column: the lower envelopes of both surfaces (EdtEnv),
//                             walked together (EdtWalk).  At a pixel of S(pred) the walk of S(target) gives s, the
//                             exact squared distance to S(target), and the other way round.  Per map: counts, the
//                             largest s, the fp64 sum of sqrt(s) and the count within the tolerance, reduced in a fixed
//                             order; the Hausdorff distance, ASSD and NSD; and every pixel's s as a key for the select
// surface_select_kernel       one CTA per map: numpy's linear percentile of each direction from
//                             the exact (lo + 1)-th and (lo + 2)-th smallest keys (block_radix_select)
//
// Every distance is sqrt(float64(s)) of an integer s < 2^25, so the only roundings are the roots, the fp64 reductions
// and the final fp32 conversion.
//
// With a spacing per map (kSp, tl_surface_distances_spaced, DESIGN §3.10) the column pass walks the weighted envelopes
// and stores each surface pixel's packed offset (edt_pack) as its key; s is the fp64 value recomputed from it, the
// maxima are taken over the bits of s (monotone as uint64 for s >= 0) and the select runs over 64-bit keys.
#pragma once
#include "edt_kernel.cuh"

namespace tl {

constexpr uint32_t kSurfNone = 0xFFFFFFFFu;  // key of a pixel off the surface: above every s
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
    uint32_t* keys;     // [2][n][H][W]: s from each pixel of S(pred) to S(target), then from S(target) to S(pred);
                        // kSurfNone off the surface
    uint32_t* stats;    // [4][n]: |S(pred)|, |S(target)|, largest s of each direction; counts 0 on a map with an
                        // empty surface, whose outputs the column pass writes in full
    int n_maps, H, W;
    double tol;         // NSD tolerance
    double qq;          // percentile / 100
    float* out;         // [4][n]: hausdorff, hausdorff_percentile, assd, nsd
    const double* spacing;  // kSp: [n][2] (sy, sx) per map; keys are then packed offsets and stats[2..3] unused
};

// kSp: max of the bits of s, as uint64
template <bool kSp>
using SurfMax = std::conditional_t<kSp, unsigned long long, uint32_t>;

template <bool kSp = false>
__global__ void __launch_bounds__(kEdtColThreads) surface_col_kernel(SurfArgs A) {
    using Env = std::conditional_t<kSp, EdtEnvW, EdtEnv>;
    using Walk = std::conditional_t<kSp, EdtWalkW, EdtWalk>;
    using Max = SurfMax<kSp>;
    __shared__ double s_red[32];
    __shared__ Max s_max[2];
    __shared__ int s_has;  // bit 0: S(pred) is nonempty, bit 1: S(target) is
    const int H = A.H, W = A.W, n = A.n_maps;
    const size_t N = (size_t)H * W, nN = (size_t)n * N;
    for (int map = blockIdx.x; map < n; map += gridDim.x) {
        if (threadIdx.x == 0) s_max[0] = s_max[1] = 0u;
        uint32_t cnt[2] = {0u, 0u}, ntol = 0u;
        Max mx[2] = {0u, 0u};
        double sum = 0.0;
        EdtSpacing spc{};
        if constexpr (kSp) spc = EdtSpacing{__ldg(A.spacing + 2 * map), __ldg(A.spacing + 2 * map + 1)};
        for (int j = threadIdx.x; j < W; j += blockDim.x) {
            Env env[2];
#pragma unroll
            for (int L = 0; L < 2; ++L) {
                env[L].col = A.h + L * nN + (size_t)map * N + j;
                env[L].stride = (size_t)W;
                env[L].top = -1;
                if constexpr (kSp) env[L].sp = spc;
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
            Walk walk[2];
#pragma unroll
            for (int L = 0; L < 2; ++L) walk[L].start(env[L], H);
            uint32_t* kp = A.keys + (size_t)map * N + j;
            uint32_t* kt = kp + nN;
            for (int u = 0; u < H; ++u) {
                // squared distances of pixel (u, j) to S(pred) and S(target): 0 exactly on that surface
                const uint32_t sp = (uint32_t)walk[0].at(env[0], u), st = (uint32_t)walk[1].at(env[1], u);
                uint32_t k0 = kSurfNone, k1 = kSurfNone;
                if constexpr (kSp) {  // a packed offset is 0 exactly at offset (0, 0), where s = 0
                    if (sp == 0u) {
                        const double s = edt_packed_sq(st, spc), d = sqrt(s);
                        k0 = st; ++cnt[0]; mx[0] = max(mx[0], (Max)__double_as_longlong(s)); sum += d;
                        ntol += d <= A.tol ? 1u : 0u;
                    }
                    if (st == 0u) {
                        const double s = edt_packed_sq(sp, spc), d = sqrt(s);
                        k1 = sp; ++cnt[1]; mx[1] = max(mx[1], (Max)__double_as_longlong(s)); sum += d;
                        ntol += d <= A.tol ? 1u : 0u;
                    }
                } else {
                    if (sp == 0u) {
                        const double d = sqrt((double)st);
                        k0 = st; ++cnt[0]; mx[0] = max(mx[0], st); sum += d; ntol += d <= A.tol ? 1u : 0u;
                    }
                    if (st == 0u) {
                        const double d = sqrt((double)sp);
                        k1 = sp; ++cnt[1]; mx[1] = max(mx[1], sp); sum += d; ntol += d <= A.tol ? 1u : 0u;
                    }
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
            Max m;
            if constexpr (kSp) {
                m = mx[L];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) m = max(m, (Max)__shfl_xor_sync(0xFFFFFFFFu, m, o));
            } else {
                m = __reduce_max_sync(0xFFFFFFFFu, mx[L]);
            }
            if ((threadIdx.x & 31) == 0) atomicMax(&s_max[L], m);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const int has = s_has;
            const float nan = __int_as_float(0x7FC00000), inf = __int_as_float(0x7F800000);
            float hd, assd, nsd;
            if (has == 3) {
                if constexpr (kSp) hd = (float)sqrt(__longlong_as_double((long long)max(s_max[0], s_max[1])));
                else hd = (float)sqrt((double)max(s_max[0], s_max[1]));
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
            if constexpr (!kSp) {
                A.stats[2 * n + map] = s_max[0];
                A.stats[3 * n + map] = s_max[1];
            }
        }
        __syncthreads();  // s_red, s_max and s_has are reused by the next map
    }
}

// numpy's linear percentile (np.percentile's default) of the cnt distances sqrt(s) whose s are the keys below kSurfNone
// of one map and direction; mx is their largest s.  The interpolation is written without FMA contraction, as numpy
// evaluates it.
__device__ __forceinline__ double surface_percentile(const uint32_t* key, int N, uint32_t cnt, uint32_t mx, double qq,
                                                     uint32_t* s_hist, uint32_t* s_digit, uint32_t* s_k,
                                                     uint32_t* s_min) {
    const double h = __dmul_rn((double)(cnt - 1u), qq);
    if (h >= (double)(cnt - 1u)) return sqrt((double)mx);
    const double lo = floor(h), g = __dsub_rn(h, lo);
    // d[lo] is the (lo + 1)-th smallest s: the (lo + 1)-th largest ~s; lo + 1 <= cnt - 1
    const RadixPick pick = block_radix_select<kSurfSelThreads>([&](int i) { return ~__ldg(key + i); }, N,
                                                               (uint32_t)lo + 1u, s_hist, s_digit, s_k);
    const uint32_t sa = ~pick.value;
    uint32_t sb = sa;
    if (pick.k >= pick.count) {  // d[lo] ends its run of equal keys: d[lo + 1] is the smallest key above it
        if (threadIdx.x == 0) *s_min = kSurfNone;
        __syncthreads();
        uint32_t m = kSurfNone;
        for (int i = threadIdx.x; i < N; i += kSurfSelThreads) {
            const uint32_t v = __ldg(key + i);
            if (v > sa) m = min(m, v);
        }
        m = __reduce_min_sync(0xFFFFFFFFu, m);
        if ((threadIdx.x & 31) == 0) atomicMin(s_min, m);
        __syncthreads();
        sb = *s_min;
        __syncthreads();  // s_min is rewritten by the next call
    }
    const double a = sqrt((double)sa), b = sqrt((double)sb), diff = __dsub_rn(b, a);
    return g >= 0.5 ? __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, g))) : __dadd_rn(a, __dmul_rn(diff, g));
}

// surface_percentile with packed-offset keys: the order is that of the fp64 s recomputed from each key, whose bits are
// monotone as uint64 (s >= 0); the sentinel sorts above every s.  h >= cnt - 1 selects the largest s (rank cnt).
__device__ __forceinline__ uint64_t surf_key64(uint32_t p, const EdtSpacing& sp) {
    return p == kSurfNone ? ~0ull : (uint64_t)__double_as_longlong(edt_packed_sq(p, sp));
}
__device__ __forceinline__ double surface_percentile_spaced(const uint32_t* key, int N, uint32_t cnt, double qq,
                                                            const EdtSpacing& sp, uint32_t* s_hist, uint32_t* s_digit,
                                                            uint32_t* s_k, unsigned long long* s_min) {
    const double h = __dmul_rn((double)(cnt - 1u), qq);
    const bool last = h >= (double)(cnt - 1u);
    const double lo = last ? (double)(cnt - 1u) : floor(h), g = __dsub_rn(h, lo);
    const RadixPickT<uint64_t> pick = block_radix_select<kSurfSelThreads, uint64_t>(
        [&](int i) { return ~surf_key64(__ldg(key + i), sp); }, N, (uint32_t)lo + 1u, s_hist, s_digit, s_k);
    const uint64_t sa = ~pick.value;
    const double a = sqrt(__longlong_as_double((long long)sa));
    if (last) return a;
    uint64_t sb = sa;
    if (pick.k >= pick.count) {  // d[lo] ends its run of equal keys: d[lo + 1] is the smallest key above it
        if (threadIdx.x == 0) *s_min = ~0ull;
        __syncthreads();
        unsigned long long m = ~0ull;
        for (int i = threadIdx.x; i < N; i += kSurfSelThreads) {
            const uint64_t v = surf_key64(__ldg(key + i), sp);
            if (v > sa) m = min(m, (unsigned long long)v);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
        if ((threadIdx.x & 31) == 0) atomicMin(s_min, m);
        __syncthreads();
        sb = *s_min;
        __syncthreads();  // s_min is rewritten by the next call
    }
    const double b = sqrt(__longlong_as_double((long long)sb)), diff = __dsub_rn(b, a);
    return g >= 0.5 ? __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, g))) : __dadd_rn(a, __dmul_rn(diff, g));
}

template <bool kSp = false>
__global__ void __launch_bounds__(kSurfSelThreads) surface_select_kernel(SurfArgs A) {
    __shared__ uint32_t s_hist[256];
    __shared__ uint32_t s_digit, s_k;
    __shared__ SurfMax<kSp> s_min;
    const int n = A.n_maps, N = A.H * A.W;
    const size_t nN = (size_t)n * N;
    for (int map = blockIdx.x; map < n; map += gridDim.x) {
        const uint32_t np = A.stats[map], nt = A.stats[n + map];
        if (np == 0u) continue;  // an empty surface: the column pass wrote this map's outputs (uniform)
        const uint32_t* kp = A.keys + (size_t)map * N;
        double pp, pt;
        if constexpr (kSp) {
            const EdtSpacing sp{__ldg(A.spacing + 2 * map), __ldg(A.spacing + 2 * map + 1)};
            pp = surface_percentile_spaced(kp, N, np, A.qq, sp, s_hist, &s_digit, &s_k, &s_min);
            pt = surface_percentile_spaced(kp + nN, N, nt, A.qq, sp, s_hist, &s_digit, &s_k, &s_min);
        } else {
            pp = surface_percentile(kp, N, np, A.stats[2 * n + map], A.qq, s_hist, &s_digit, &s_k, &s_min);
            pt = surface_percentile(kp + nN, N, nt, A.stats[3 * n + map], A.qq, s_hist, &s_digit, &s_k, &s_min);
        }
        if (threadIdx.x == 0) A.out[n + map] = (float)fmax(pp, pt);
    }
}

}  // namespace tl
