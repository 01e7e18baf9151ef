// Topological prior loss (Clough et al., IPMI 2019 / TPAMI 2022) on the sorted persistence pairs of tl_diagrams_*:
// per map, the beta largest persistences are pushed towards 1 and the rest towards 0 (tl_prior_forward /
// tl_prior_backward).
//
// prior_cost_kernel      one CTA per map: p_r = |f[des_r] - f[cre_r]| of each record of the map's diagram (gudhi
//                        emission order, as tl_diagrams_gather hands it out), an exact block-wide radix select of the
//                        beta-th largest key (p bits << 32 | ~position), the per-map threshold key and the cost
//                        sum_{rank < beta} (1 - p^2) + sum_{rank >= beta} p^2 + max(0, beta - count), fp64, fixed order
// prior_backward_kernel  one CTA per map: zero fill, then each record's key is recomputed, compared with the stored
//                        threshold and its gradient scatter-added into the creator and destroyer pixels
//
// Ranking by the 64-bit key is "p descending, ties by position, earlier first": a stable descending sort.  p is never
// negative, so its bits order like its values; the low word ~position makes every key of a map distinct.
#pragma once
#include "tl_common.cuh"

namespace tl {

constexpr int kPriorThreads = 512;
constexpr int kPriorWarps = kPriorThreads / 32;
// threshold keys: a record is selected iff its key >= the map's threshold.  Keys stay below 2^63 (fabsf clears the
// sign bit), so these two never select anything.
constexpr uint64_t kPriorNone = 0xFFFFFFFFFFFFFFFFull;     // beta = 0
constexpr uint64_t kPriorInvalid = 0xFFFFFFFFFFFFFFFEull;  // negative beta or a status bit: cost and gradient NaN

struct PriorArgs {
    const PairRec* arena;      // sorted records of every map (sorted_pairs)
    const uint32_t* offs;      // [n_maps] first record of each map
    const int32_t* counts;     // [n_maps] records of each map
    const float* maps;         // [n_maps][N]: the values (read from the maps, so -0.0 survives)
    long long N;
    int n_maps;
    const int32_t* betti;      // [n_maps]
    const unsigned int* status;
    uint32_t* pbits;           // scratch, parallel to the arena: p bits of each record
    uint64_t* thr;             // [n_maps] threshold key (kept in the state for the backward)
    float* cost;               // [n_maps]
};

__device__ __forceinline__ float prior_diff(const float* f, const PairRec& r) { return __ldg(f + r.des) - __ldg(f + r.cre); }

__global__ void __launch_bounds__(kPriorThreads) prior_cost_kernel(PriorArgs A) {
    __shared__ uint32_t s_hist[256];
    __shared__ uint32_t s_digit, s_k, s_idx;
    __shared__ uint32_t s_warp[kPriorWarps];
    __shared__ double s_red[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool bad_status = *A.status != 0u;
    for (int map = blockIdx.x; map < A.n_maps; map += gridDim.x) {
        const int beta = A.betti[map];
        if (bad_status || beta < 0) {
            if (tid == 0) { A.cost[map] = __int_as_float(0x7FC00000); A.thr[map] = kPriorInvalid; }
            continue;  // uniform across the block
        }
        const int n = A.counts[map];
        const PairRec* recs = A.arena + A.offs[map];
        const float* f = A.maps + (size_t)map * A.N;
        uint32_t* pb = A.pbits + A.offs[map];
        for (int i = tid; i < n; i += kPriorThreads) pb[i] = __float_as_uint(fabsf(prior_diff(f, recs[i])));
        uint64_t thr;
        if (beta == 0) {
            thr = kPriorNone;
        } else if (beta >= n) {
            thr = 0ull;  // every record
        } else {
            __syncthreads();  // pb is complete
            // 1. radix select of the beta-th largest p bits; prefix / k are uniform
            const RadixPick pick = block_radix_select<kPriorThreads>([&](int i) { return pb[i]; }, n, (uint32_t)beta,
                                                                     s_hist, &s_digit, &s_k);
            const uint32_t prefix = pick.value, k = pick.k;
            // 2. among the records with p bits == prefix, the k-th in position order is the last one selected
            if (tid == 0) s_idx = 0xFFFFFFFFu;
            uint32_t run = 0u;
            for (int i0 = 0; i0 < n; i0 += kPriorThreads) {
                const int i = i0 + tid;
                const bool eq = i < n && pb[i] == prefix;
                const unsigned bal = __ballot_sync(0xFFFFFFFFu, eq);
                if (lane == 0) s_warp[warp] = (uint32_t)__popc(bal);
                __syncthreads();
                uint32_t before = run, chunk = 0u;
                for (int w = 0; w < kPriorWarps; ++w) { const uint32_t s = s_warp[w]; if (w < warp) before += s; chunk += s; }
                if (eq && before + (uint32_t)__popc(bal & lanemask_lt()) + 1u == k) s_idx = (uint32_t)i;
                run += chunk;
                __syncthreads();
                if (s_idx != 0xFFFFFFFFu) break;  // uniform
            }
            thr = ((uint64_t)prefix << 32) | (uint64_t)(~s_idx);
        }
        __syncthreads();  // every pb[i] is visible to the thread that sums it (beta == 0 / beta >= n skipped the barrier)
        // 3. the cost, each thread over a fixed stride, then the fixed-order block sum
        double acc = 0.0;
        for (int i = tid; i < n; i += kPriorThreads) {
            const uint32_t v = pb[i];
            const double p = (double)__uint_as_float(v);
            const double p2 = p * p;
            const uint64_t key = ((uint64_t)v << 32) | (uint64_t)(~(uint32_t)i);
            acc += key >= thr ? 1.0 - p2 : p2;
        }
        const double s = block_sum(acc, s_red);
        if (tid == 0) {
            A.cost[map] = (float)(s + (double)(beta > n ? beta - n : 0));
            A.thr[map] = thr;
        }
        __syncthreads();  // s_red, s_idx are reused by the next map
    }
}

struct PriorBwdArgs {
    const PairRec* arena;
    const uint32_t* offs;
    const int32_t* counts;
    const float* maps;
    int N, n_maps;
    const uint64_t* thr;
    const unsigned int* status;
    const float* grad_cost;    // [n_maps]
    float* grad_maps;          // [n_maps][N], fully overwritten
};

// One CTA per map, as diagram_backward_kernel.  d cost / d death = -2 (d - b) for a selected record, +2 (d - b)
// otherwise, and the opposite for the birth; a map whose cost was NaN (negative beta, status bit) gets NaN everywhere.
__global__ void __launch_bounds__(512) prior_backward_kernel(PriorBwdArgs A) {
    const bool bad_status = *A.status != 0u;
    for (int map = blockIdx.x; map < A.n_maps; map += gridDim.x) {
        const uint64_t thr = A.thr[map];
        const bool bad = bad_status || thr == kPriorInvalid;
        const float fill = bad ? __int_as_float(0x7FC00000) : 0.f;
        float* g = A.grad_maps + (size_t)map * A.N;
        if (((reinterpret_cast<uintptr_t>(g) & 15) == 0) && (A.N & 3) == 0) {
            float4* g4 = reinterpret_cast<float4*>(g);
            for (int i = threadIdx.x; i < (A.N >> 2); i += blockDim.x) g4[i] = make_float4(fill, fill, fill, fill);
        } else {
            for (int i = threadIdx.x; i < A.N; i += blockDim.x) g[i] = fill;
        }
        if (bad) continue;  // uniform across the block
        __syncthreads();  // the fill is visible to the whole CTA before its atomics land on the same lines
        const int n = A.counts[map];
        const PairRec* recs = A.arena + A.offs[map];
        const float* f = A.maps + (size_t)map * A.N;
        const float gc = __ldg(A.grad_cost + map);
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const PairRec r = recs[i];
            const float diff = prior_diff(f, r);
            const uint64_t key = ((uint64_t)__float_as_uint(fabsf(diff)) << 32) | (uint64_t)(~(uint32_t)i);
            const float t = 2.f * diff * gc;  // d (d - b)^2 / d d, times the upstream gradient
            const float gd = key >= thr ? -t : t;
            if ((unsigned int)r.cre < (unsigned int)A.N) atomicAdd(g + r.cre, -gd);
            if ((unsigned int)r.des < (unsigned int)A.N) atomicAdd(g + r.des, gd);
        }
        __syncthreads();
    }
}

}  // namespace tl
