// Persistence diagrams and the Wasserstein cost as differentiable building blocks (tl_diagrams_*,
// tl_wasserstein_backward): the pieces torch_topological's CubicalComplex / WassersteinDistance hand to
// autograd, for losses composed in Python instead of the fused tl_forward.
//
// diagram_offsets_kernel   exclusive scan of the per-map pair counts the persistence launch left in the
//                          workspace -> offsets[n_maps + 1], plus a copy of the status word
// diagram_gather_kernel    pairs[P][2] (creator, destroyer) and diagram[P][2] = (f[creator], f[destroyer]),
//                          packed by map in gudhi's emission order
// diagram_backward_kernel  grad_maps = scatter-add of grad_diagram into the critical pixels (IndexBackward)
// wasserstein_backward_kernel  d cost_k / d (birth, death) of both diagrams of pair k, from the matching
#pragma once
#include "tl_common.cuh"

namespace tl {

constexpr int kScanThreads = 1024;

// One CTA: offsets[i] = sum of counts[0 .. i), offsets[n_maps] = total; *status_out = *status.
__global__ void __launch_bounds__(kScanThreads) diagram_offsets_kernel(const int32_t* __restrict__ counts, int n_maps,
                                                                         const unsigned int* __restrict__ status,
                                                                         int32_t* __restrict__ offsets, int32_t* __restrict__ status_out) {
    __shared__ int32_t s_warp[kScanThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int32_t carry = 0;  // the host capped the record count below 2^31
    for (int base = 0; base < n_maps; base += kScanThreads) {
        const int i = base + tid;
        const int32_t v = i < n_maps ? counts[i] : 0;
        int32_t incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int32_t before = 0, chunk = 0;
        for (int w = 0; w < kScanThreads / 32; ++w) { const int32_t s = s_warp[w]; if (w < warp) before += s; chunk += s; }
        if (i < n_maps) offsets[i] = carry + before + incl - v;
        carry += chunk;
        __syncthreads();  // s_warp is rewritten by the next chunk
    }
    if (tid == 0) {
        offsets[n_maps] = carry;
        if (status_out) *status_out = (int32_t)*status;
    }
}

// One CTA per map (grid-stride).  The values are read from the map itself rather than from the records: the
// records of the shared-memory kernel carry values that went through the sort key (mono32 / unmono32), which
// turns -0.0 into +0.0, and the diagram must equal x.ravel()[pairs] bit for bit.
__global__ void __launch_bounds__(256) diagram_gather_kernel(const PairRec* __restrict__ arena, const uint32_t* __restrict__ rec_off,
                                                             const float* __restrict__ maps, long long N, int n_maps,
                                                             const int32_t* __restrict__ offsets, int2* __restrict__ pairs,
                                                             float2* __restrict__ diagram) {
    for (int map = blockIdx.x; map < n_maps; map += gridDim.x) {
        const int o = offsets[map], n = offsets[map + 1] - o;
        const PairRec* recs = arena + rec_off[map];
        const float* f = maps + (size_t)map * N;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const PairRec r = recs[i];
            pairs[o + i] = make_int2(r.cre, r.des);
            diagram[o + i] = make_float2(__ldg(f + r.cre), __ldg(f + r.des));
        }
    }
}

// One CTA per map, as grad_one_map: zero-fill the map's gradient, then scatter-add.  A pixel can be critical for
// several pairs (a creator of one, the destroyer of another); the atomics add those up.  Indices outside the map
// are skipped.
__global__ void __launch_bounds__(512) diagram_backward_kernel(const int2* __restrict__ pairs, const int32_t* __restrict__ offsets,
                                                               const float2* __restrict__ grad_diagram, int n_maps, int N,
                                                               float* __restrict__ grad_maps) {
    for (int map = blockIdx.x; map < n_maps; map += gridDim.x) {
        float* g = grad_maps + (size_t)map * N;
        if (((reinterpret_cast<uintptr_t>(g) & 15) == 0) && (N & 3) == 0) {
            float4* g4 = reinterpret_cast<float4*>(g);
            for (int i = threadIdx.x; i < (N >> 2); i += blockDim.x) g4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
            for (int i = threadIdx.x; i < N; i += blockDim.x) g[i] = 0.f;
        }
        __syncthreads();  // the fill is visible to the whole CTA before its atomics land on the same lines
        const int o0 = offsets[map], o1 = offsets[map + 1];
        for (int i = o0 + threadIdx.x; i < o1; i += blockDim.x) {
            const int2 p = pairs[i];
            const float2 gd = grad_diagram[i];
            if ((unsigned int)p.x < (unsigned int)N) atomicAdd(g + p.x, gd.x);
            if ((unsigned int)p.y < (unsigned int)N) atomicAdd(g + p.y, gd.y);
        }
        __syncthreads();
    }
}

// d M / d (b, d) of one diagram point, the formula of pair_gradient (grad_kernel.cuh) without the loss_r term and
// without the coefficient: matched to (tb, td): cdist(p=inf) backward (the full gradient on both coordinates at an
// exact tie, zero at distance 0) after .pow(q); matched to the diagonal: (-1/2, +1/2) * d/dx x^q of the distance
// x = (d - b) / 2, with 1 at x == 0 for q == 1 as pow's backward gives.
__device__ __forceinline__ void point_gradient_diag(float b, float d, double q, double& gb, double& gd) {
    const float h = 0.5f * (b + d);
    const float x = fmaxf(fabsf(b - h), fabsf(d - h));
    const double gg = x > 0.f ? (q == 2.0 ? 2.0 * (double)x : q * pow((double)x, q - 1.0)) : (q == 1.0 ? 1.0 : 0.0);
    const double s = d > b ? 1.0 : (d < b ? -1.0 : 0.0);
    gb = -0.5 * gg * s; gd = 0.5 * gg * s;
}
__device__ __forceinline__ void point_gradient_matched(float b, float d, float tb, float td, double q, double& gb, double& gd) {
    const float xb = b - tb, xd = d - td, ab = fabsf(xb), ad = fabsf(xd);
    const float dist = fmaxf(ab, ad);
    const double gg = dist > 0.f ? q * pow((double)dist, q - 1.0) : 0.0;
    gb = ab == dist ? gg * (xb > 0.f ? 1.0 : (xb < 0.f ? -1.0 : 0.0)) : 0.0;
    gd = ad == dist ? gg * (xd > 0.f ? 1.0 : (xd < 0.f ? -1.0 : 0.0)) : 0.0;
}

struct WassersteinBwdArgs {
    const float2* d1; const int32_t* off1;
    const float2* d2; const int32_t* off2;
    int n_diag;
    float q;
    const int32_t* match1;     // tl_wasserstein's matching: row of diagram k of D2, or -1 for the diagonal
    const float* grad_cost;    // [n_diag] upstream gradient of each cost
    float2* g1; float2* g2;    // either may be null
};

// One CTA per diagram pair.  D2's rows first get the diagonal term, then the pass over D1's rows overwrites the
// rows its points are matched to with the negated matched term: the inverse matching is never stored, and each
// matched row of D2 is written by exactly one thread (the matching is one-to-one).
__global__ void __launch_bounds__(256) wasserstein_backward_kernel(WassersteinBwdArgs A) {
    const double q = (double)A.q;
    for (int k = blockIdx.x; k < A.n_diag; k += gridDim.x) {
        const int o1 = A.off1[k], n1 = A.off1[k + 1] - o1;
        const int o2 = A.off2[k], n2 = A.off2[k + 1] - o2;
        const double gc = (double)__ldg(A.grad_cost + k);
        if (A.g2) {
            for (int j = threadIdx.x; j < n2; j += blockDim.x) {
                const float2 p = A.d2[o2 + j];
                double gb, gd;
                point_gradient_diag(p.x, p.y, q, gb, gd);
                A.g2[o2 + j] = make_float2((float)(gb * gc), (float)(gd * gc));
            }
            __syncthreads();  // the diagonal terms are in place before matched rows overwrite them
        }
        for (int i = threadIdx.x; i < n1; i += blockDim.x) {
            const float2 p = A.d1[o1 + i];
            const int m = A.match1[o1 + i];
            double gb, gd;
            if (m >= 0 && m < n2) {
                const float2 t = A.d2[o2 + m];
                point_gradient_matched(p.x, p.y, t.x, t.y, q, gb, gd);
                gb *= gc; gd *= gc;
                if (A.g2) A.g2[o2 + m] = make_float2((float)(-gb), (float)(-gd));
            } else {
                point_gradient_diag(p.x, p.y, q, gb, gd);
                gb *= gc; gd *= gc;
            }
            if (A.g1) A.g1[o1 + i] = make_float2((float)gb, (float)gd);
        }
        __syncthreads();
    }
}

}  // namespace tl
