// Exact Euclidean distance transform of 2-D binary maps (tl_edt), the Hausdorff distance-transform loss
// (tl_hausdorff_dt_*), and the signed distance map and boundary loss (tl_signed_distance, tl_boundary_*).
// Separable, in the style of Meijster et al. (2000) / Felzenszwalb & Huttenlocher (2012):
//
// edt_row_kernel<Src, NL>   one warp per row: per pixel, the horizontal distance h_L to the nearest pixel of label L
//                           in its row (kEdtNone if the row has none), from 32-pixel ballots; NL = 1: label 0 only
//                           (uint32 per pixel), NL = 2: labels 0 and 1 (uint2 per pixel)
// edt_col_kernel<Mode, M>   one CTA per map, one thread per column: per label, the lower envelope of the parabolas
//                           (u - i)^2 + h_i^2 over the rows i with a finite h_i, built top to bottom with its stack
//                           stored in place over the column's h words, then queried top to bottom: the exact squared
//                           distance s of every pixel to the nearest pixel of that label
// hausdorff_dt_backward_kernel  elementwise: d cost / d x from the field D saved by the forward
// edt_col_kernel<kEdtSigned>    the signed distance map phi (tl_signed_distance) and the boundary loss's cost
//                               (tl_boundary_forward); boundary_backward_kernel: d cost / d x from the saved phi
//
// Every quantity of the envelope is an integer below 2^26 (H, W <= 4096: s <= 2 * 4095^2), so int32 holds all of it
// and no float enters before the final root.  Entry point checks keep H and W in [1, 4096].
//
// With a physical pixel spacing (sy, sx) per map (a non-null spacing, DESIGN §3.10) the row pass is the same, and the
// column pass builds the weighted envelope (metric EdtSpacing, not EdtUnit): row i's parabola is the fp64 value
// s(u) = (float64(u - i) * sy)^2 + (float64(h_i) * sx)^2, each operation rounded, and the walk yields the offset
// (|u - v|, h) of the nearest pixel, packed in 24 bits (edt_pack), from which s is recomputed where it is needed.
#pragma once
#include <type_traits>
#include "tl_common.cuh"

namespace tl {

constexpr uint32_t kEdtNone = 0xFFFFFFFFu;  // h of a row without a pixel of the label
constexpr int kEdtMaxDim = 4096;
constexpr int kEdtRowWarps = 8;
constexpr int kEdtColThreads = 256;

// p = torch.sigmoid(x) for fp32 exactly as PyTorch's CUDA kernel evaluates it (1 / (1 + exp(-x)), IEEE division,
// no fast-math), so that p > 0.5 is the same predicate as torch.sigmoid(x) > 0.5 at every input, NaN included
__device__ __forceinline__ float edt_sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

struct EdtMaskSrc {    // tl_edt: a nonzero byte is label 1
    const uint8_t* m;
    __device__ __forceinline__ bool operator()(size_t i) const { return __ldg(m + i) != 0; }
};
struct EdtLogitSrc {   // P = sigmoid(x) > 0.5
    const float* x;
    __device__ __forceinline__ bool operator()(size_t i) const { return edt_sigmoid(__ldg(x + i)) > 0.5f; }
};
struct EdtTargetSrc {  // T = t > 0.5
    const float* t;
    __device__ __forceinline__ bool operator()(size_t i) const { return __ldg(t + i) > 0.5f; }
};

// rows: n_rows rows of W pixels; out: n_rows * W words (NL = 1) or uint2 (NL = 2)
template <class Src, int NL>
__global__ void __launch_bounds__(kEdtRowWarps * 32) edt_row_kernel(Src src, long long n_rows, int W, uint32_t* out) {
    constexpr int kChunks = kEdtMaxDim / 32;
    __shared__ uint32_t s_bal[kEdtRowWarps][NL][kChunks];  // ballot of label L over chunk c
    __shared__ int s_right[kEdtRowWarps][NL][kChunks];     // first pixel of label L right of chunk c (or a sentinel)
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int nc = (W + 31) >> 5;
    const unsigned lt = lanemask_lt(), le = lt | (1u << lane);
    constexpr int kFar = 1 << 24;  // farther than any pixel: a distance to it never wins
    for (long long row = (long long)blockIdx.x * kEdtRowWarps + wib; row < n_rows; row += (long long)gridDim.x * kEdtRowWarps) {
        const size_t base = (size_t)row * W;
        for (int c = 0; c < nc; ++c) {
            const int j = c * 32 + lane;
            const bool in = j < W;
            const bool lab = in && src(base + j);
            const unsigned b0 = __ballot_sync(0xFFFFFFFFu, in && !lab);
            const unsigned b1 = __ballot_sync(0xFFFFFFFFu, lab);
            if (lane == 0) {
                s_bal[wib][0][c] = b0;
                if (NL == 2) s_bal[wib][NL - 1][c] = b1;
            }
        }
        __syncwarp();
        if (lane == 0) {
            int r[NL];
#pragma unroll
            for (int L = 0; L < NL; ++L) r[L] = kFar;
            for (int c = nc - 1; c >= 0; --c) {
#pragma unroll
                for (int L = 0; L < NL; ++L) {
                    s_right[wib][L][c] = r[L];
                    const unsigned b = s_bal[wib][L][c];
                    if (b) r[L] = c * 32 + __ffs(b) - 1;
                }
            }
        }
        __syncwarp();
        int left[NL];
#pragma unroll
        for (int L = 0; L < NL; ++L) left[L] = -kFar;
        for (int c = 0; c < nc; ++c) {
            const int j = c * 32 + lane;
            uint32_t h[NL];
#pragma unroll
            for (int L = 0; L < NL; ++L) {
                const unsigned b = s_bal[wib][L][c];
                const unsigned bl = b & le, br = b & ~lt;
                const int pl = bl ? c * 32 + 31 - __clz(bl) : left[L];
                const int pr = br ? c * 32 + __ffs(br) - 1 : s_right[wib][L][c];
                const int d = min(j - pl, pr - j);
                h[L] = d < kFar / 2 ? (uint32_t)d : kEdtNone;
                if (b) left[L] = c * 32 + 31 - __clz(b);
            }
            if (j < W) {
                if (NL == 1) out[base + j] = h[0];
                else reinterpret_cast<uint2*>(out)[base + j] = make_uint2(h[0], h[NL - 1]);
            }
        }
        __syncwarp();  // s_bal / s_right are rewritten for the next row
    }
}

__device__ __forceinline__ int edt_ceil_div(int a, int b) { return a >= 0 ? (a + b - 1) / b : -((-a) / b); }

// The first integer u at which the parabola of row i (horizontal distance hi) is <= that of row v < i:
// (u - i)^2 + hi^2 <= (u - v)^2 + hv^2  <=>  2u (i - v) >= i^2 + hi^2 - v^2 - hv^2.  |numerator| < 2^26.
__device__ __forceinline__ int edt_sep(int v, int hv, int i, int hi) {
    return edt_ceil_div(i * i + hi * hi - v * v - hv * hv, 2 * (i - v));
}

// ---- the weighted parabolas (physical spacing)

// float64(d) * sp, squared, each operation rounded to fp64 (no contraction)
__device__ __forceinline__ double edt_sq1(int d, double sp) {
    const double a = __dmul_rn((double)d, sp);
    return __dmul_rn(a, a);
}

// a1 + b1 <= a2 + b2 for doubles, exactly as real numbers: a rounded sum orders the reals (round to nearest is
// monotone), and on equal rounded sums the exact rounding errors (TwoSum) decide
__device__ __forceinline__ double edt_two_sum_err(double a, double b, double s) {
    const double t = __dsub_rn(s, a);
    return __dadd_rn(__dsub_rn(a, __dsub_rn(s, t)), __dsub_rn(b, t));
}
__device__ __forceinline__ bool edt_sum_le(double a1, double b1, double a2, double b2) {
    const double s1 = __dadd_rn(a1, b1), s2 = __dadd_rn(a2, b2);
    if (s1 != s2) return s1 < s2;
    return edt_two_sum_err(a1, b1, s1) <= edt_two_sum_err(a2, b2, s2);
}

// Row i (horizontal term bi = edt_sq1(hi, sx)) is <= row v (bv) at u, in the exact sums of the rounded terms.  For
// i > v the set of u where this holds is a suffix of [0, H) (DESIGN §3.10)
__device__ __forceinline__ bool edt_beats(int i, double bi, int v, double bv, int u, double sy) {
    return edt_sum_le(edt_sq1(abs(u - i), sy), bi, edt_sq1(abs(u - v), sy), bv);
}

// The first u in [0, H] at which row i > v beats row v (H: none): the crossing of the exact parabolas as an fp64
// estimate, then corrected by the exact predicate, which is monotone in u, so the answer does not depend on the estimate
__device__ __forceinline__ int edt_sep_w(int v, int hv, int i, int hi, int H, double sy, double sx) {
    const double bv = edt_sq1(hv, sx), bi = edt_sq1(hi, sx);
    // the estimate only has to land near the answer, so fp32 does (|error| << 1 wherever it is in [0, H]); the fp64
    // division or reciprocal would bring a slow-path call, which spills
    const float est = 0.5f * (float)(i + v) + __fdividef((float)(bi - bv), (float)(2.0 * (double)(i - v) * (sy * sy)));
    int u = (int)fminf(fmaxf(ceilf(est), 0.f), (float)H);
    while (u > 0 && edt_beats(i, bi, v, bv, u - 1, sy)) --u;
    while (u < H && !edt_beats(i, bi, v, bv, u, sy)) ++u;
    return u;
}

// offsets below 4096 each, packed in 24 bits; 0 exactly at offset (0, 0)
__device__ __forceinline__ uint32_t edt_pack(int dy, int dx) { return (uint32_t)dy | ((uint32_t)dx << 12); }

// ---- the metric of the column pass
//
// What differs between unit and physical spacing.  EdtUnit: the integer parabolas; the walk yields s itself.
// EdtSpacing: the weighted parabolas of the map's spacing; the walk yields the packed offset (|u - v|, h) of the nearest
// pixel (edt_pack), from which s is recomputed where it is needed.  Each metric gives
//   sep(v, hv, i, hi, H)          the first u at which row i > v is <= row v (EdtSpacing: in [0, H], H for none)
//   at(dy, h)                     what the walk yields at row offset dy = u - v and distance h; 0 exactly at (0, 0)
//   sq(e)                         the fp64 squared distance s of a walk value
//   key(e), key_sq(k)             walk values as unsigned integers in the order of s, kEdtNone above all of them,
//                                 and the fp64 s of a key

struct EdtUnit {
    using Key = uint32_t;
    static __device__ __forceinline__ EdtUnit of(const double*, int) { return {}; }
    __device__ __forceinline__ int sep(int v, int hv, int i, int hi, int) const { return edt_sep(v, hv, i, hi); }
    __device__ __forceinline__ int at(int dy, int h) const { return dy * dy + h * h; }
    __device__ __forceinline__ double sq(int s) const { return (double)s; }
    __device__ __forceinline__ Key key(uint32_t s) const { return s; }
    __device__ __forceinline__ double key_sq(Key k) const { return (double)k; }
};

struct EdtSpacing {
    using Key = unsigned long long;  // the bits of s, monotone as uint64 for s >= 0
    double sy, sx;                   // size of a pixel along rows (dim -2) and along columns (dim -1)
    static __device__ __forceinline__ EdtSpacing of(const double* spacing, int map) {
        return {__ldg(spacing + 2 * map), __ldg(spacing + 2 * map + 1)};
    }
    __device__ __forceinline__ int sep(int v, int hv, int i, int hi, int H) const { return edt_sep_w(v, hv, i, hi, H, sy, sx); }
    __device__ __forceinline__ uint32_t at(int dy, int h) const { return edt_pack(abs(dy), h); }
    // the squared distance of offset (dy, dx) as scipy's distance_transform_edt(sampling=...) evaluates it
    __device__ __forceinline__ double sq(uint32_t p) const {
        return __dadd_rn(edt_sq1((int)(p & 0xFFFu), sy), edt_sq1((int)(p >> 12), sx));
    }
    __device__ __forceinline__ Key key(uint32_t p) const { return p == kEdtNone ? ~0ull : (Key)__double_as_longlong(sq(p)); }
    __device__ __forceinline__ double key_sq(Key k) const { return __longlong_as_double((long long)k); }
};

// The lower envelope of one label over one column.  Entry k of the stack (row v_k, distance h_k, packed v | h << 16)
// lives in the column's word of row k: when row i is pushed the stack holds at most i + 1 entries, and rows <= i have
// been read, so the stack only overwrites consumed input.  The start z_k of entry k (the first u it is the minimum at;
// z_0 = 0) is recomputed from entries k - 1 and k when it is needed.
template <class Metric>
struct EdtEnv {
    uint32_t* col;
    size_t stride;
    int top, v, h, z;  // top entry and its start; top = -1: empty
    Metric m;

    __device__ __forceinline__ void load(int k, int& vk, int& hk) const {
        const uint32_t e = col[(size_t)k * stride];
        vk = (int)(e & 0xFFFFu);
        hk = (int)(e >> 16);
    }
    __device__ __forceinline__ void put(int k, int vk, int hk) { col[(size_t)k * stride] = (uint32_t)vk | ((uint32_t)hk << 16); }

    __device__ __forceinline__ void push(int i, int hi, int H) {
        while (top >= 0) {
            // Row i against the top: pushed from its start s if that is below H, skipped if it never is the
            // minimum, or else the top is popped.  Written once per metric: folded into one metric method, the test
            // cost either a spill in the unit signed-map kernel or about 1% of the weighted Hausdorff DT loss (B200).
            if constexpr (std::is_same_v<Metric, EdtUnit>) {
                const int s = edt_sep(v, h, i, hi);
                if (s > z) {  // row i is the minimum from s on; past the last row it never is
                    if (s < H) { put(++top, i, hi); v = i; h = hi; z = s; }
                    return;
                }
            } else {
                // the pop test and the skip test are single comparisons at the top's start and at the last row; the
                // separator (with its division) is only computed for an entry that is pushed
                const double bi = edt_sq1(hi, m.sx), bv = edt_sq1(h, m.sx);
                if (!edt_beats(i, bi, v, bv, z, m.sy)) {
                    if (edt_beats(i, bi, v, bv, H - 1, m.sy)) {
                        const int s = m.sep(v, h, i, hi, H);
                        put(++top, i, hi); v = i; h = hi; z = s;
                    }
                    return;
                }
            }
            if (--top >= 0) {  // row i is <= the top over the top's whole range: pop it
                load(top, v, h);
                if (top == 0) {
                    z = 0;
                } else {
                    int pv, ph;
                    load(top - 1, pv, ph);
                    z = m.sep(pv, ph, v, h, H);
                }
            }
        }
        top = 0;
        put(0, i, hi);
        v = i; h = hi; z = 0;
    }
};

// Walks an envelope top to bottom: the walk value of the nearest pixel for u = 0, 1, ..., H - 1 in that order.
template <class Metric>
struct EdtWalk {
    int k, top, v, h, nv, nh, znext, H;
    __device__ __forceinline__ void start(const EdtEnv<Metric>& e, int H_) {
        top = e.top; H = H_; k = 0;
        if (top < 0) return;
        e.load(0, v, h);
        znext = H;
        if (top >= 1) { e.load(1, nv, nh); znext = e.m.sep(v, h, nv, nh, H); }
    }
    __device__ __forceinline__ auto at(const EdtEnv<Metric>& e, int u) {
        while (u >= znext) {
            ++k; v = nv; h = nh; znext = H;
            if (k < top) { e.load(k + 1, nv, nh); znext = e.m.sep(v, h, nv, nh, H); }
        }
        return e.m.at(u - v, h);
    }
};

// kEdtSigned: the signed distance map phi of the boundary loss (DESIGN §3.11) and, given logits, its cost
enum EdtMode { kEdtField = 0, kEdtPred = 1, kEdtTarget = 2, kEdtSigned = 3 };

// s^(alpha / 2) = F^alpha in fp64
__device__ __forceinline__ double edt_pow(double d, double half_alpha) {
    return half_alpha == 1.0 ? d : half_alpha == 0.5 ? sqrt(d) : d == 0.0 ? 0.0 : exp(half_alpha * log(d));
}

struct EdtColArgs {
    uint32_t* h;            // row pass output: [n][H][W] words (kEdtField) or uint2 (kEdtPred, kEdtTarget, kEdtSigned)
    int n_maps, H, W;
    float* field;           // kEdtField: out [n][H][W]; kEdtSigned: phi [n][H][W]
    int32_t* sp;            // kEdtPred: s of P per pixel (0 where P is not mixed), in the D buffer
    float* D;               // kEdtTarget: F(P)^a + F(T)^a, overwriting sp
    const float* x;         // kEdtTarget: logits; kEdtSigned: logits, or null for phi alone
    const float* t;         // kEdtTarget: targets
    double half_alpha;
    float* cost;            // kEdtTarget, kEdtSigned with x: [n]
    const double* spacing;  // EdtSpacing: [n][2] (sy, sx) per map
    double inv_hw;          // kEdtSigned with x: 1 / HW (a device fp64 division would bring a slow-path call that spills)
};

// Metric: EdtUnit, or EdtSpacing of each map's spacing; sp then holds the packed offset of P's nearest other-label pixel
template <int Mode, class Metric>
__global__ void __launch_bounds__(kEdtColThreads) edt_col_kernel(EdtColArgs A) {
    constexpr int NL = Mode == kEdtField ? 1 : 2;
    __shared__ double s_red[32];
    const int H = A.H, W = A.W;
    const size_t N = (size_t)H * W;
    for (int map = blockIdx.x; map < A.n_maps; map += gridDim.x) {
        double acc = 0.0;
        const Metric m = Metric::of(A.spacing, map);
        for (int j = threadIdx.x; j < W; j += blockDim.x) {
            EdtEnv<Metric> env[NL];
#pragma unroll
            for (int L = 0; L < NL; ++L) {
                env[L].col = A.h + ((size_t)map * N + j) * NL + L;
                env[L].stride = (size_t)W * NL;
                env[L].top = -1;
                env[L].m = m;
            }
            for (int i = 0; i < H; ++i) {
#pragma unroll
                for (int L = 0; L < NL; ++L) {
                    const uint32_t hi = env[L].col[(size_t)i * env[L].stride];
                    if (hi != kEdtNone) env[L].push(i, (int)hi, H);
                }
            }
            EdtWalk<Metric> walk[NL];
#pragma unroll
            for (int L = 0; L < NL; ++L) walk[L].start(env[L], H);
            const size_t o = (size_t)map * N + j;
            if (Mode == kEdtField) {
                // the same loop in two shapes, each the one that compiles tightest for its metric: testing the empty
                // envelope per pixel takes EdtUnit fewer registers than hoisting the test, and hoisting it keeps
                // EdtSpacing from spilling around sqrt's slow path
                if constexpr (std::is_same_v<Metric, EdtUnit>) {
                    for (int u = 0; u < H; ++u)
                        A.field[o + (size_t)u * W] = env[0].top < 0 ? __int_as_float(0x7F800000)
                                                                    : (float)sqrt(m.sq(walk[0].at(env[0], u)));
                } else if (env[0].top < 0) {
                    for (int u = 0; u < H; ++u) A.field[o + (size_t)u * W] = __int_as_float(0x7F800000);
                } else {
                    for (int u = 0; u < H; ++u) A.field[o + (size_t)u * W] = (float)sqrt(m.sq(walk[0].at(env[0], u)));
                }
            } else if constexpr (Mode == kEdtSigned) {
                // label 0 is the background: on a mixed map s1 == 0 exactly on the foreground, where phi = 1 - d_in
                // (d_in = sqrt(s0)); elsewhere phi = d_out = sqrt(s1).  fp64, rounded once; __dsub_rn / __dmul_rn /
                // __dadd_rn keep nvcc from contracting (DESIGN §3.11)
                const bool mixed = env[0].top >= 0 && env[1].top >= 0;
                for (int u = 0; u < H; ++u) {
                    const size_t q = o + (size_t)u * W;
                    float phi = 0.f;
                    if (mixed) {  // the walk value is 0 exactly at the label's own pixels
                        const auto e0 = walk[0].at(env[0], u), e1 = walk[1].at(env[1], u);
                        const double d = sqrt(m.sq(e1 == 0 ? e0 : e1));
                        phi = (float)(e1 == 0 ? __dsub_rn(1.0, d) : d);
                    }
                    A.field[q] = phi;
                    if (A.x) acc = __dadd_rn(acc, __dmul_rn((double)edt_sigmoid(__ldg(A.x + q)), (double)phi));
                }
            } else {
                // a map with both labels: exactly one of s0, s1 is 0 per pixel; with one label only the field is 0
                const bool mixed = env[0].top >= 0 && env[1].top >= 0;
                for (int u = 0; u < H; ++u) {
                    const size_t q = o + (size_t)u * W;
                    const int s = mixed ? walk[0].at(env[0], u) + walk[1].at(env[1], u) : 0;
                    if (Mode == kEdtPred) {
                        A.sp[q] = s;
                    } else {
                        const double d = edt_pow(m.sq(A.sp[q]), A.half_alpha) + edt_pow(m.sq(s), A.half_alpha);
                        const double p = (double)edt_sigmoid(__ldg(A.x + q)), diff = p - (double)__ldg(A.t + q);
                        acc += diff * diff * d;
                        A.D[q] = (float)d;
                    }
                }
            }
        }
        if (Mode == kEdtTarget || (Mode == kEdtSigned && A.x)) {
            const double s = block_sum(acc, s_red);
            if (threadIdx.x == 0) A.cost[map] = Mode == kEdtTarget ? (float)(s / (double)N) : (float)__dmul_rn(s, A.inv_hw);
            __syncthreads();  // s_red is reused by the next map
        }
    }
}

// grad_x = grad_cost[map] * (2 / HW) * (p - t) * D * p (1 - p), fp64, rounded to fp32; blocks of 1024 pixels
__global__ void __launch_bounds__(256) hausdorff_dt_backward_kernel(const float* x, const float* t, const float* D,
                                                                     const float* grad_cost, int n_maps, long long N,
                                                                     float* grad) {
    const long long per_map = (N + 1023) / 1024;
    for (long long b = blockIdx.x; b < (long long)n_maps * per_map; b += gridDim.x) {
        const int map = (int)(b / per_map);
        const long long lo = (b - (long long)map * per_map) * 1024, hi = min(lo + 1024, N);
        const double scale = 2.0 * (double)__ldg(grad_cost + map) / (double)N;
        const size_t base = (size_t)map * N;
        for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
            const double p = (double)edt_sigmoid(__ldg(x + base + i));
            grad[base + i] = (float)(scale * (p - (double)__ldg(t + base + i)) * (double)__ldg(D + base + i) * p * (1.0 - p));
        }
    }
}

// the boundary loss: grad_x = grad_cost[map] * (1 / HW) * phi * p (1 - p), fp64, rounded to fp32, from the phi saved by
// the forward (recomputing it would repeat the transform); blocks of 1024 pixels
__global__ void __launch_bounds__(256) boundary_backward_kernel(const float* x, const float* phi, const float* grad_cost,
                                                                 int n_maps, long long N, float* grad) {
    const long long per_map = (N + 1023) / 1024;
    for (long long b = blockIdx.x; b < (long long)n_maps * per_map; b += gridDim.x) {
        const int map = (int)(b / per_map);
        const long long lo = (b - (long long)map * per_map) * 1024, hi = min(lo + 1024, N);
        const double scale = (double)__ldg(grad_cost + map) / (double)N;
        const size_t base = (size_t)map * N;
        for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
            const double p = (double)edt_sigmoid(__ldg(x + base + i));
            grad[base + i] = (float)(scale * (double)__ldg(phi + base + i) * p * (1.0 - p));
        }
    }
}

}  // namespace tl
