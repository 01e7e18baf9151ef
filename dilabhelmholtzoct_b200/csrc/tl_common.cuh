// Shared device helpers for the topological-loss kernels (sm_100a).
//
// Geometry and ordering follow the gudhi cubical complex the reference reaches through
// torch_topological (reference call site /root/reference/octsam/models/topological_loss.py:55-63;
// cell semantics in SURVEY.md section 8a-note):
//   * pixels are the 2-cells of a (2H+1)x(2W+1) bitmap; an edge/vertex takes the min of its cofaces;
//   * total order of cells: (value, dimension, bitmap position);
//   * H0 = elder-rule union-find on the vertex graph, edges ascending;
//   * H1 = elder-rule union-find on the dual graph (squares + OUTSIDE), edges descending
//     (2-D Alexander duality).
// Both are expressed in ONE ascending form: for H1 every key is bit-complemented, so
// "smaller key" always means "earlier in the scan" (edges) / "elder" (nodes).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace tl {

struct __align__(8) PairRec {
    int32_t cre, des;  // creator / destroyer pixel (flat r*W+c)
    float b, d;        // diagram point gathered from the map: (f[cre], f[des])
    float tb, td;      // matched ground-truth point, NaN = matched to the diagonal (pred side only)
};

// Device status word (workspace header): sticky bits set by the kernels, folded into the loss as NaN and
// readable through tl_status().  With the default (typical-size) workspace a pathological input can
// exhaust the pair arena or, on maps of more than 65536 pixels, the basin tables; the worst-case
// workspace (tl_set_option(TL_OPT_WORST_CASE_WORKSPACE, 1)) cannot overflow.
constexpr unsigned int kStArena = 1u;      // pair arena exhausted: some maps lost pairs
constexpr unsigned int kStBasins = 2u;     // more basins than the per-CTA tables hold (multi-band maps)
constexpr unsigned int kStNonFinite = 4u;  // a map holds a NaN: the pairing is undefined

// Where persistence pairs live: ONE record arena shared by all maps of both sets, carved with a device
// counter (a map's pairs are contiguous; maps land in the order they finish), instead of a worst-case
// stride of H*W/2 records per map.
struct PairStore {
    PairRec* arena;
    uint64_t* skeys;               // sort key per record (death-cell order), parallel to arena; may be null
    unsigned long long* head;      // next free record
    unsigned long long cap;        // records in the arena
    uint32_t* offs[2];             // [n_maps] first record of each map
    int32_t* counts[2];            // [n_maps] records of each map
    double* dsum[2];               // [n_maps] sum over the map's points of their cost to the diagonal
    unsigned int* status;
    float q;                       // exponent of the Wasserstein cost (for dsum)
};

__device__ __forceinline__ float powq(float x, float q) { return q == 2.0f ? x * x : powf(x, q); }
// torch.cdist(p=inf) entry, then .pow(q)
__device__ __forceinline__ float cost_pp(float b, float d, float b2, float d2, float q) {
    return powq(fmaxf(fabsf(b - b2), fabsf(d - d2)), q);
}
// torch.linalg.vector_norm(D - 0.5*(x+y), inf), then .pow(q)
__device__ __forceinline__ float cost_diag(float b, float d, float q) {
    const float h = 0.5f * (b + d);
    return powq(fmaxf(fabsf(b - h), fabsf(d - h)), q);
}

// deterministic block-wide sum (shuffle tree per warp, then the warps in order); s_red: 32 doubles
__device__ __forceinline__ double block_sum(double x, double* s_red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xFFFFFFFFu, x, o);
    __syncthreads();
    if (lane == 0) s_red[warp] = x;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += s_red[w];
    return t;
}

// Reserve `total` records for one map (one thread calls this): returns the first record and how many
// of them fit; an exhausted arena sets the status bit and truncates.
__device__ __forceinline__ unsigned long long ps_reserve(const PairStore& ps, int set, int map, int total, int* avail) {
    const unsigned long long base = total > 0 ? atomicAdd(ps.head, (unsigned long long)total) : 0ull;
    int a = total;
    if (base + (unsigned long long)total > ps.cap) {
        a = base < ps.cap ? (int)(ps.cap - base) : 0;
        atomicOr(ps.status, kStArena);
    }
    ps.offs[set][map] = (uint32_t)(base < ps.cap ? base : 0ull);
    ps.counts[set][map] = a;
    *avail = a;
    return base;
}

__device__ __forceinline__ uint32_t mono32(float f) {
    uint32_t u = __float_as_uint(f);
    if (u == 0x80000000u) u = 0u;  // -0.0 == +0.0 in the reference's double compare
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// inverse of mono32 (exact; the two zeros both come back as +0.0)
__device__ __forceinline__ float unmono32(uint32_t m) {
    return __uint_as_float((m & 0x80000000u) ? (m & 0x7FFFFFFFu) : ~m);
}

// L2 residency hints (per instruction, no device-wide state): the map a CTA works on is read three times (level 0,
// compaction, emission) and should stay in L2 between them; the pair records are written once and read by later
// kernels only, so they stream past it.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_normal() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// 128-bit store with an L2 eviction policy
__device__ __forceinline__ void stg_v4_hint(void* ptr, uint4 v, uint64_t policy) {
    asm volatile("st.global.L2::cache_hint.v4.b32 [%0], {%1,%2,%3,%4}, %5;" :: "l"(ptr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(policy) : "memory");
}
// The 128-byte line at `ptr` (128-byte aligned) holds nothing anybody will read again: L2 may drop it without
// writing it back to DRAM
__device__ __forceinline__ void l2_discard_line(const void* ptr) {
    asm volatile("discard.global.L2 [%0], 128;" :: "l"(ptr) : "memory");
}
__device__ __forceinline__ float4 ldg_f4_keep(const float4* ptr, uint64_t policy) {
    float4 v;
    asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(ptr), "l"(policy));
    return v;
}

__device__ __forceinline__ uint64_t ld_cg_u64(const uint64_t* p) {
    return __ldcg(reinterpret_cast<const unsigned long long*>(p));
}

__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// The digit of the k-th largest (1-based) among the 256 bins of s_hist, scanning from digit 255 down.  Warp 0 only;
// lane l owns digits 255 - 8l .. 248 - 8l.  Writes the digit and k minus the count of larger digits.
__device__ __forceinline__ void radix_pick_digit(const uint32_t* s_hist, uint32_t k, uint32_t* s_digit, uint32_t* s_k) {
    const int lane = threadIdx.x & 31;
    uint32_t c[8], sum = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) { c[j] = s_hist[255 - 8 * lane - j]; sum += c[j]; }
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
    uint32_t run = incl - sum;
    if (run < k && k <= incl) {  // exactly one lane
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (run + c[j] >= k) { *s_digit = (uint32_t)(255 - 8 * lane - j); *s_k = k - run; break; }
            run += c[j];
        }
    }
}

template <class T>
struct RadixPickT {
    T value;         // the k-th largest value
    uint32_t k;      // its rank (1-based) among the values equal to it
    uint32_t count;  // how many values equal it
};
using RadixPick = RadixPickT<uint32_t>;

// Exact block-wide radix select of the k-th largest (1 <= k <= n) of the n keys key(0) .. key(n - 1) (T = uint32_t:
// 4 passes, uint64_t: 8), 8 bits per pass from the top.  Every thread of a kThreads-thread block calls it with the
// same n and k; the trip counts are uniform, so whole warps reach __match_any_sync.  s_hist is 256 words of shared
// memory, s_digit and s_k one word each; the last barrier leaves them free for the caller.  For the k-th smallest,
// select over ~key.
template <int kThreads, class T = uint32_t, class Key>
__device__ __forceinline__ RadixPickT<T> block_radix_select(const Key& key, int n, uint32_t k, uint32_t* s_hist,
                                                            uint32_t* s_digit, uint32_t* s_k) {
    constexpr int kTop = 8 * (int)sizeof(T) - 8;
    const int tid = threadIdx.x, lane = tid & 31;
    T prefix = 0u;
    uint32_t count = 0u;
    for (int shift = kTop; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += kThreads) s_hist[i] = 0u;
        __syncthreads();
        const T hi_mask = shift == kTop ? (T)0u : ~(T)0u << (shift + 8);
        for (int i0 = 0; i0 < n; i0 += kThreads) {
            const int i = i0 + tid;
            uint32_t d = 256u + (uint32_t)lane;  // distinct dummy digit for lanes without a candidate
            if (i < n) {
                const T v = key(i);
                if ((v & hi_mask) == prefix) d = (uint32_t)(v >> shift) & 255u;
            }
            const unsigned peers = __match_any_sync(0xFFFFFFFFu, d);
            if (d < 256u && (peers & lanemask_lt()) == 0u) atomicAdd(&s_hist[d], (uint32_t)__popc(peers));
        }
        __syncthreads();
        if ((tid >> 5) == 0) radix_pick_digit(s_hist, k, s_digit, s_k);
        __syncthreads();
        prefix |= (T)*s_digit << shift;
        k = *s_k;
        count = s_hist[*s_digit];
        __syncthreads();  // s_hist / s_digit / s_k are rewritten by the next pass or the caller
    }
    return RadixPickT<T>{prefix, k, count};
}

// Exact n / d for n < 2^24, d <= 8193 via multiply-shift (magic = ceil(2^40 / d)); avoids the
// ~30-instruction integer division in the per-node / per-edge loops.
struct FastDiv {
    uint64_t magic;
    uint32_t d;
    __host__ __device__ explicit FastDiv(uint32_t d_) : magic(((1ull << 40) + d_ - 1) / d_), d(d_) {}
    __host__ __device__ FastDiv(uint64_t magic_, uint32_t d_) : magic(magic_), d(d_) {}  // magic computed by the host
    __host__ __device__ static uint64_t magic_of(uint32_t d_) { return ((1ull << 40) + d_ - 1) / d_; }
    __device__ __forceinline__ uint32_t div(uint32_t n) const { return (uint32_t)(((uint64_t)n * magic) >> 40); }
};

// Triplet-table entry: high 32 bits = merge code, low 32 bits = target node.
//   code 0            : level-0 link (merged before every recorded edge; always followed)
//   code 0xFFFFFFFF   : root (never merged)
//   otherwise         : bitmap position of the merging edge + 1
constexpr uint32_t kCodeL0 = 0u;
constexpr uint32_t kCodeRoot = 0xFFFFFFFFu;

template <int DIM>
struct Geo {
    const float* f;
    int H, W, GW, VW, NN, OUT;

    __device__ __forceinline__ Geo(const float* f_, int H_, int W_)
        : f(f_), H(H_), W(W_), GW(2 * W_ + 1), VW(W_ + 1),
          NN(DIM == 1 ? H_ * W_ + 1 : (H_ + 1) * (W_ + 1)), OUT(H_ * W_) {}

    __device__ __forceinline__ float px(int r, int c) const { return __ldg(f + r * W + c); }

    // v-edge(i,j): between pixels (i,j-1),(i,j), j in [0,W]; h-edge(i,j): between (i-1,j),(i,j), i in [0,H]
    __device__ __forceinline__ float vedge_val(int i, int j) const {
        if (j == 0) return px(i, 0);
        if (j == W) return px(i, W - 1);
        return fminf(px(i, j - 1), px(i, j));
    }
    __device__ __forceinline__ float hedge_val(int i, int j) const {
        if (i == 0) return px(0, j);
        if (i == H) return px(H - 1, j);
        return fminf(px(i - 1, j), px(i, j));
    }
    __device__ __forceinline__ int vedge_top(int i, int j) const {
        if (j == 0) return i * W;
        if (j == W) return i * W + W - 1;
        float a = px(i, j - 1), b = px(i, j);
        return a <= b ? i * W + j - 1 : i * W + j;  // left pixel if it attains the min
    }
    __device__ __forceinline__ int hedge_top(int i, int j) const {
        if (i == 0) return j;
        if (i == H) return (H - 1) * W + j;
        float a = px(i - 1, j), b = px(i, j);
        return a <= b ? (i - 1) * W + j : i * W + j;  // upper pixel if it attains the min
    }
    // vertex (i,j): min over the <=4 surrounding pixels and the first raster pixel attaining it
    __device__ __forceinline__ float vertex_val(int i, int j, int* top) const {
        float best = 0.f;
        int bi = -1;
#pragma unroll
        for (int di = -1; di <= 0; ++di)
#pragma unroll
            for (int dj = -1; dj <= 0; ++dj) {
                int r = i + di, c = j + dj;
                if (r < 0 || r >= H || c < 0 || c >= W) continue;
                float v = px(r, c);
                if (bi < 0 || v < best) { best = v; bi = r * W + c; }
            }
        if (top) *top = bi;
        return best;
    }

    __device__ __forceinline__ uint64_t make_ekey(float val, uint32_t pos) const {
        uint64_t k = ((uint64_t)mono32(val) << 32) | pos;
        return DIM == 1 ? ~k : k;
    }
    __device__ __forceinline__ float edge_val(uint32_t pos) const {
        int Y = pos / GW, X = pos - Y * GW;
        return (Y & 1) ? vedge_val(Y >> 1, X >> 1) : hedge_val(Y >> 1, X >> 1);
    }
    __device__ __forceinline__ uint64_t ekey(uint32_t pos) const { return make_ekey(edge_val(pos), pos); }
    __device__ __forceinline__ int edge_top(uint32_t pos) const {
        int Y = pos / GW, X = pos - Y * GW;
        return (Y & 1) ? vedge_top(Y >> 1, X >> 1) : hedge_top(Y >> 1, X >> 1);
    }
    // node key: smaller = elder
    __device__ __forceinline__ uint64_t nkey(int x) const {
        if (DIM == 1) {
            if (x == OUT) return 0ull;
            return ~(((uint64_t)mono32(__ldg(f + x)) << 32) | (uint32_t)x);
        } else {
            int i = x / VW, j = x - i * VW;
            return ((uint64_t)mono32(vertex_val(i, j, nullptr)) << 32) | (uint32_t)x;
        }
    }
};

}  // namespace tl
