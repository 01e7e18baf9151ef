// Betti matching of prediction / target map pairs (Stucki et al., ICML 2023, "Topologically faithful image
// segmentation via induced matching of persistence barcodes"): tl_betti_*.
//
// For a prediction map L, a target map G and the comparison image C = min(L, G) (formed on the fly, never stored),
// one CTA per map pair runs four elder-rule merge trees on the pixel graph of the T-construction (tl_common.cuh):
//
//   run 0  L -> L   the barcode of L          node keys from L, edge keys from L
//   run 1  G -> G   the barcode of G
//   run 2  L -> C   the image barcode of H_d(L_t) -> H_d(C_t)
//   run 3  G -> C
//
// Image persistence by union-find.  H0: nodes are vertices keyed by the DOMAIN, edges are scanned in the CODOMAIN
// order; a node dies at the first codomain edge that joins it to a node with a smaller domain key, which is the
// pivot structure of the boundary matrix with columns in the codomain order and rows in the domain order (Cohen-
// Steiner, Edelsbrunner, Harer and Morozov, SODA 2009; Bauer and Schmahl, SoCG 2023): every vertex is a row from the
// start, so the elder rule compares all nodes of a codomain component, present in L_t or not.  H1 is the same
// union-find on the dual graph (squares + OUTSIDE, edges descending) of the anti-transposed matrix: the inclusion
// reverses, so the node keys come from the CODOMAIN squares and the edges in the DOMAIN order; a dying square is the
// death cell in C and its edge the birth cell in the domain.  An image interval is kept when birth < death strictly.
// With domain == codomain the runs are the ordinary barcode (cubical_persistence's pairs).
//
// Each run: (a) every node links to the far end of its EARLIEST incident edge when that end is elder -- exact,
// because before that edge the node is alone, and the component it joins has a root at least as old as the far end;
// (b) pointer jumping flattens those links (the far end's own earliest edge comes no later than the shared edge, so
// each replaced fact "x joins elder z at level e_x" still holds); (c) every other edge goes through the lock-free
// triplet merge tree of ph_kernel.cuh (the correctness argument there does not use any relation between node and
// edge keys); (d) the per-node result is written to an int32 table.  Unlike ph_kernel.cuh's level-0 contraction,
// (a) records the real edge, so it stays exact when node and edge keys come from different maps.
//
// Matching: an L interval and a G interval are matched when their image intervals (which share their BIRTH cell)
// die at the same cell of C -- an edge for H0, a square for H1; the two essential H0 classes are always matched.
// Records of a map: the intervals of L in the order of the node that owns them (H0: birth vertex, H1: death square,
// raster order), matched and unmatched split into two lists; the essential H0 pair last among the matched; the
// unmatched intervals of G in the same order.
#pragma once
#include "tl_common.cuh"

namespace tl {

constexpr int kBmThreads = 1024;
constexpr uint32_t kCodePre = 0x80000000u;  // flag on a link of step (a); positions stay below 2^31 (check_shape)

struct BettiArgs {
    const float* pred;            // [n_maps][H*W]
    const float* target;
    int n_maps, H, W;
    unsigned int* job_counter;
    unsigned long long* head;     // next free record of the arena
    unsigned long long cap;       // records in the arena
    int4* arena;                  // matched (pc, pd, tc, td) | unmatched pred (pc, pd, -, -) | unmatched target (tc, td, -, -)
    uint32_t* recoff;             // [n_maps] first record of each map
    int32_t* counts;              // [3][n_maps]: matched, unmatched pred, unmatched target
    float* cost;                  // [n_maps]
    unsigned int* status;
    uint64_t* T;                  // per slot: [t_stride] merge tree
    int32_t* tabs;                // per slot: 6 node tables [n_stride] + 2 edge tables [e_stride]
    size_t t_stride, tab_stride, n_stride, e_stride;
};

// pixel source: one map, or the pixelwise minimum of two (the comparison image)
struct Pix {
    const float* a;
    const float* b;
    __device__ __forceinline__ float operator()(int p) const {
        const float v = __ldg(a + p);
        return b ? fminf(v, __ldg(b + p)) : v;
    }
};

template <int DIM>
struct BGeo {
    Pix np, ep;  // node keys from np, edge keys from ep
    int H, W, GW, VW, NN, OUT;

    __device__ __forceinline__ BGeo(Pix n, Pix e, int H_, int W_)
        : np(n), ep(e), H(H_), W(W_), GW(2 * W_ + 1), VW(W_ + 1),
          NN(DIM == 1 ? H_ * W_ + 1 : (H_ + 1) * (W_ + 1)), OUT(H_ * W_) {}

    __device__ __forceinline__ float edge_val(uint32_t pos) const {
        const int Y = (int)(pos / (uint32_t)GW), X = (int)pos - Y * GW;
        const int i = Y >> 1, j = X >> 1;
        if (Y & 1) return j == 0 ? ep(i * W) : (j == W ? ep(i * W + W - 1) : fminf(ep(i * W + j - 1), ep(i * W + j)));
        return i == 0 ? ep(j) : (i == H ? ep((H - 1) * W + j) : fminf(ep((i - 1) * W + j), ep(i * W + j)));
    }
    __device__ __forceinline__ uint64_t ekey(uint32_t pos) const {
        const uint64_t k = ((uint64_t)mono32(edge_val(pos)) << 32) | pos;
        return DIM == 1 ? ~k : k;
    }
    // DIM 0: the vertex value (min of its <= 4 pixels); DIM 1: the pixel (x != OUT)
    __device__ __forceinline__ float node_val(int x) const {
        if (DIM == 1) return np(x);
        const int i = x / VW, j = x - i * VW;
        float best = __int_as_float(0x7F800000);
        if (i > 0 && j > 0) best = fminf(best, np((i - 1) * W + j - 1));
        if (i > 0 && j < W) best = fminf(best, np((i - 1) * W + j));
        if (i < H && j > 0) best = fminf(best, np(i * W + j - 1));
        if (i < H && j < W) best = fminf(best, np(i * W + j));
        return best;
    }
    __device__ __forceinline__ uint64_t nkey(int x) const {  // smaller = elder
        if (DIM == 1) return x == OUT ? 0ull : ~(((uint64_t)mono32(np(x)) << 32) | (uint32_t)x);
        return ((uint64_t)mono32(node_val(x)) << 32) | (uint32_t)x;
    }
    // the interval stored at node x with edge `pos` is non-empty: birth < death strictly
    __device__ __forceinline__ bool positive(int x, uint32_t pos) const {
        const uint32_t e = mono32(edge_val(pos)), n = mono32(node_val(x));
        return DIM == 0 ? n < e : e < n;
    }
    // compact edge index: v-edges (i, j) first, then h-edges
    __device__ __forceinline__ int eidx(uint32_t pos) const {
        const int Y = (int)(pos / (uint32_t)GW), X = (int)pos - Y * GW;
        return (Y & 1) ? (Y >> 1) * VW + (X >> 1) : H * VW + (Y >> 1) * W + (X >> 1);
    }

    __device__ static __forceinline__ uint32_t pos_of(uint32_t code) { return (code & ~kCodePre) - 1u; }

    // representative of x at level skey: follow entries merged at or before skey
    __device__ __forceinline__ int rep(const uint64_t* T, int x, uint64_t skey, uint64_t& entry) const {
        for (;;) {
            const uint64_t t = ld_cg_u64(T + x);
            const uint32_t code = (uint32_t)(t >> 32);
            if (code == kCodeRoot || ekey(pos_of(code)) > skey) { entry = t; return x; }
            x = (int)(uint32_t)t;
        }
    }

    // triplet-merge-tree Merge(a, edge, b), lock-free (ph_kernel.cuh, Ph::merge)
    __device__ void merge(uint64_t* T, int a, int b, uint32_t pos, uint64_t skey) const {
        uint32_t code = pos + 1;
        for (;;) {
            uint64_t ta, tb;
            int x = rep(T, a, skey, ta), y = rep(T, b, skey, tb);
            if (x == y) return;
            if (nkey(y) < nkey(x)) { const int t = x; x = y; y = t; tb = ta; }
            const unsigned long long want = ((unsigned long long)code << 32) | (uint32_t)x;
            const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(T + y), (unsigned long long)tb, want);
            if (old == tb) {
                const uint32_t ocode = (uint32_t)(tb >> 32);
                if (ocode == kCodeRoot) return;
                a = x; b = (int)(uint32_t)tb; code = ocode; skey = ekey(pos_of(ocode));
            } else {
                a = x; b = y;
            }
        }
    }
};

// one run: out[x] = bitmap position of the edge at which node x's non-empty interval ends (H0) / begins (H1), -1
// otherwise; the root's index goes to *root
template <int DIM>
__device__ void betti_run(const BGeo<DIM>& g, uint64_t* T, int32_t* out, int* root) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const int H = g.H, W = g.W, GW = g.GW, VW = g.VW, NN = g.NN;
    for (int x = tid; x < NN; x += nt) T[x] = ((uint64_t)kCodeRoot << 32) | (uint32_t)x;
    __syncthreads();
    // (a) earliest incident edge, linked when its far end is elder
    const int n_real = DIM == 1 ? H * W : NN;
    for (int x = tid; x < n_real; x += nt) {
        uint64_t best = ~0ull;
        int other = -1;
        auto consider = [&](uint32_t pos, int o) {
            const uint64_t k = g.ekey(pos);
            if (k < best) { best = k; other = o; }
        };
        if (DIM == 1) {
            const int r = x / W, c = x - r * W;
            consider((uint32_t)(2 * c + 1 + (2 * r) * GW), r == 0 ? g.OUT : x - W);
            consider((uint32_t)(2 * c + 1 + (2 * r + 2) * GW), r == H - 1 ? g.OUT : x + W);
            consider((uint32_t)(2 * c + (2 * r + 1) * GW), c == 0 ? g.OUT : x - 1);
            consider((uint32_t)(2 * c + 2 + (2 * r + 1) * GW), c == W - 1 ? g.OUT : x + 1);
        } else {
            const int i = x / VW, j = x - i * VW;
            if (i > 0) consider((uint32_t)(2 * j + (2 * i - 1) * GW), x - VW);
            if (i < H) consider((uint32_t)(2 * j + (2 * i + 1) * GW), x + VW);
            if (j > 0) consider((uint32_t)(2 * j - 1 + (2 * i) * GW), x - 1);
            if (j < W) consider((uint32_t)(2 * j + 1 + (2 * i) * GW), x + 1);
        }
        if (other >= 0 && g.nkey(other) < g.nkey(x)) {
            const uint32_t pos = DIM == 1 ? (uint32_t)~best : (uint32_t)best;
            T[x] = ((uint64_t)((pos + 1) | kCodePre) << 32) | (uint32_t)other;
        }
    }
    __syncthreads();
    // (b) flatten the links of (a) by pointer jumping (own entry only)
    for (;;) {
        int changed = 0;
        for (int x = tid; x < n_real; x += nt) {
            const uint64_t t = ld_cg_u64(T + x);
            if ((uint32_t)(t >> 32) == kCodeRoot) continue;
            const uint64_t tp = ld_cg_u64(T + (uint32_t)t);
            if ((uint32_t)(tp >> 32) != kCodeRoot) { T[x] = (t & 0xFFFFFFFF00000000ull) | (tp & 0xFFFFFFFFull); changed = 1; }
        }
        if (!__syncthreads_or(changed)) break;
    }
    // (c) every edge into the triplet merge tree; an edge whose ends hang under one root of (a) is inside that tree
    const int n_vedges = H * (W + 1), n_edges = n_vedges + (H + 1) * W;
    for (int e = tid; e < n_edges; e += nt) {
        int a, b;
        uint32_t pos;
        if (e < n_vedges) {
            const int i = e / (W + 1), j = e - i * (W + 1);
            pos = (uint32_t)(2 * j + (2 * i + 1) * GW);
            if (DIM == 1) { a = j == 0 ? g.OUT : i * W + j - 1; b = j == W ? g.OUT : i * W + j; }
            else { a = i * VW + j; b = a + VW; }
        } else {
            const int e2 = e - n_vedges, i = e2 / W, j = e2 - i * W;
            pos = (uint32_t)(2 * j + 1 + (2 * i) * GW);
            if (DIM == 1) { a = i == 0 ? g.OUT : (i - 1) * W + j; b = i == H ? g.OUT : i * W + j; }
            else { a = i * VW + j; b = a + 1; }
        }
        // links of (a) never change during (c): representatives are always roots of (a)
        const uint64_t ta = ld_cg_u64(T + a), tb = ld_cg_u64(T + b);
        const uint32_t ca = (uint32_t)(ta >> 32), cb = (uint32_t)(tb >> 32);
        const int la = ca != kCodeRoot && (ca & kCodePre) ? (int)(uint32_t)ta : a;
        const int lb = cb != kCodeRoot && (cb & kCodePre) ? (int)(uint32_t)tb : b;
        if (la != lb) g.merge(T, la, lb, pos, g.ekey(pos));
    }
    __syncthreads();
    // (d) per-node result
    for (int x = tid; x < NN; x += nt) {
        const uint64_t t = ld_cg_u64(T + x);
        const uint32_t code = (uint32_t)(t >> 32);
        int32_t v = -1;
        if (code == kCodeRoot) {
            if (DIM == 0) *root = x;  // one root: the graph is connected
        } else {
            const uint32_t pos = BGeo<DIM>::pos_of(code);
            if (g.positive(x, pos)) v = (int32_t)pos;
        }
        out[x] = v;
    }
    __syncthreads();
}

// creator / destroyer pixels of the barcode interval of map f stored at node x with edge pos
template <int DIM>
__device__ __forceinline__ int2 interval_pixels(const float* f, int H, int W, int x, uint32_t pos) {
    const Geo<DIM> g(f, H, W);
    int2 r;
    if (DIM == 0) { g.vertex_val(x / g.VW, x % g.VW, &r.x); r.y = g.edge_top(pos); }
    else { r.x = g.edge_top(pos); r.y = x; }
    return r;
}

__device__ __forceinline__ double sq(double x) { return x * x; }

template <int DIM>
__global__ void __launch_bounds__(kBmThreads) betti_kernel(BettiArgs A) {
    __shared__ unsigned int s_job;
    __shared__ int s_flag, s_root[2], s_cnt[3];
    __shared__ unsigned long long s_argmax[2], s_base;
    __shared__ int s_w[2][kBmThreads / 32];
    __shared__ double s_red[kBmThreads / 32];
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const int H = A.H, W = A.W, N = H * W;
    uint64_t* T = A.T + (size_t)blockIdx.x * A.t_stride;
    int32_t* tabs = A.tabs + (size_t)blockIdx.x * A.tab_stride;
    int32_t* P[2] = {tabs, tabs + A.n_stride};                     // barcode of L / G
    int32_t* I[2] = {tabs + 2 * A.n_stride, tabs + 3 * A.n_stride};  // image L -> C / G -> C
    int32_t* part[2] = {tabs + 4 * A.n_stride, tabs + 5 * A.n_stride};  // partner node in the other map, or -1
    int32_t* tab[2] = {tabs + 6 * A.n_stride, tabs + 6 * A.n_stride + A.e_stride};

    for (;;) {
        __syncthreads();
        if (tid == 0) {
            s_job = atomicAdd(A.job_counter, 1u);
            s_flag = 0; s_root[0] = s_root[1] = 0; s_cnt[0] = s_cnt[1] = s_cnt[2] = 0; s_argmax[0] = s_argmax[1] = 0ull;
        }
        __syncthreads();
        const unsigned int job = s_job;
        if (job >= (unsigned)A.n_maps) break;
        const int map = (int)job;
        const float* L = A.pred + (size_t)map * N;
        const float* G = A.target + (size_t)map * N;
        {   // NaN check (the order is undefined) and argmax, first in raster order (the H0 essential destroyer)
            unsigned long long best[2] = {0ull, 0ull};
            bool has_nan = false;
            for (int p = tid; p < N; p += nt) {
                const float lv = __ldg(L + p), gv = __ldg(G + p);
                has_nan |= lv != lv || gv != gv;
                const unsigned long long lo = (uint32_t)(0xFFFFFFFFu - (uint32_t)p);
                const unsigned long long kl = ((unsigned long long)mono32(lv) << 32) | lo, kg = ((unsigned long long)mono32(gv) << 32) | lo;
                best[0] = kl > best[0] ? kl : best[0];
                best[1] = kg > best[1] ? kg : best[1];
            }
            if (DIM == 0) { atomicMax(&s_argmax[0], best[0]); atomicMax(&s_argmax[1], best[1]); }
            if (has_nan) s_flag = 1;
        }
        __syncthreads();
        if (s_flag) {  // block-uniform
            if (tid == 0) {
                atomicOr(A.status, kStNonFinite);
                for (int k = 0; k < 3; ++k) A.counts[k * A.n_maps + map] = 0;
                A.recoff[map] = 0;
                A.cost[map] = __int_as_float(0x7FC00000);
            }
            continue;
        }
        const Pix pl{L, nullptr}, pg{G, nullptr}, pc{L, G};
        betti_run<DIM>(BGeo<DIM>(pl, pl, H, W), T, P[0], &s_root[0]);
        betti_run<DIM>(BGeo<DIM>(pg, pg, H, W), T, P[1], &s_root[1]);
        int dummy;
        if (DIM == 0) {
            betti_run<DIM>(BGeo<DIM>(pl, pc, H, W), T, I[0], &dummy);
            betti_run<DIM>(BGeo<DIM>(pg, pc, H, W), T, I[1], &dummy);
        } else {
            betti_run<DIM>(BGeo<DIM>(pc, pl, H, W), T, I[0], &dummy);
            betti_run<DIM>(BGeo<DIM>(pc, pg, H, W), T, I[1], &dummy);
        }
        const BGeo<DIM> geo(pl, pl, H, W);  // geometry only
        const int NN = geo.NN, n_edges = H * (W + 1) + (H + 1) * W;
        for (int x = tid; x < NN; x += nt) { part[0][x] = -1; part[1][x] = -1; }
        for (int e = tid; e < n_edges; e += nt) { tab[0][e] = -1; tab[1][e] = -1; }
        __syncthreads();
        // H0: death edge in C -> node of the image interval; H1: birth edge -> node of the barcode interval
        for (int x = tid; x < NN; x += nt)
            for (int s = 0; s < 2; ++s) {
                const int32_t v = DIM == 0 ? I[s][x] : P[s][x];
                if (v >= 0) tab[s][geo.eidx((uint32_t)v)] = x;
            }
        __syncthreads();
        for (int x = tid; x < NN; x += nt) {
            if (DIM == 0) {
                for (int s = 0; s < 2; ++s) {
                    if (P[s][x] < 0 || I[s][x] < 0) continue;
                    const int32_t o = tab[1 - s][geo.eidx((uint32_t)I[s][x])];
                    if (o >= 0 && P[1 - s][o] >= 0) part[s][x] = o;
                }
            } else if (I[0][x] >= 0 && I[1][x] >= 0) {  // x: a square of C at which both image intervals die
                const int32_t z = tab[0][geo.eidx((uint32_t)I[0][x])], zg = tab[1][geo.eidx((uint32_t)I[1][x])];
                if (z >= 0 && zg >= 0) { part[0][z] = zg; part[1][zg] = z; }
            }
        }
        __syncthreads();
        {   // counts
            int c[3] = {0, 0, 0};
            for (int x = tid; x < NN; x += nt) {
                if (P[0][x] >= 0) ++c[part[0][x] >= 0 ? 0 : 1];
                if (P[1][x] >= 0 && part[1][x] < 0) ++c[2];
            }
            for (int k = 0; k < 3; ++k) {
                const int v = __reduce_add_sync(0xFFFFFFFFu, c[k]);
                if (lane == 0 && v) atomicAdd(&s_cnt[k], v);
            }
        }
        __syncthreads();
        const int n_m = s_cnt[0] + (DIM == 0 ? 1 : 0), n_p = s_cnt[1], n_t = s_cnt[2];
        if (tid == 0) {
            const unsigned long long total = (unsigned long long)(n_m + n_p + n_t);
            const unsigned long long base = atomicAdd(A.head, total);
            int ok = base + total <= A.cap;
            if (!ok) atomicOr(A.status, kStArena);
            A.counts[map] = ok ? n_m : 0;
            A.counts[A.n_maps + map] = ok ? n_p : 0;
            A.counts[2 * A.n_maps + map] = ok ? n_t : 0;
            A.recoff[map] = ok ? (uint32_t)base : 0u;
            s_base = base;
            s_flag = ok ? 0 : 2;
        }
        __syncthreads();
        if (s_flag) { if (tid == 0) A.cost[map] = __int_as_float(0x7FC00000); continue; }
        int4* out = A.arena + s_base;
        double acc = 0.0;
        // L's intervals in node order: matched rows from 0, unmatched rows from n_m
        int base_m = 0, base_p = 0;
        for (int x0 = 0; x0 < NN; x0 += nt) {
            const int x = x0 + tid;
            const int32_t pos = x < NN ? P[0][x] : -1;
            const int32_t z = pos >= 0 ? part[0][x] : -1;
            const bool m = pos >= 0 && z >= 0, u = pos >= 0 && z < 0;
            const unsigned bm = __ballot_sync(0xFFFFFFFFu, m), bu = __ballot_sync(0xFFFFFFFFu, u);
            if (lane == 0) { s_w[0][warp] = __popc(bm); s_w[1][warp] = __popc(bu); }
            __syncthreads();
            int before_m = 0, tot_m = 0, before_u = 0, tot_u = 0;
            for (int w = 0; w < kBmThreads / 32; ++w) {
                const int vm = s_w[0][w], vu = s_w[1][w];
                tot_m += vm; tot_u += vu;
                if (w < warp) { before_m += vm; before_u += vu; }
            }
            if (m || u) {
                const int2 pp = interval_pixels<DIM>(L, H, W, x, (uint32_t)pos);
                const double b = __ldg(L + pp.x), d = __ldg(L + pp.y);
                if (m) {
                    const int2 tp = interval_pixels<DIM>(G, H, W, z, (uint32_t)P[1][z]);
                    out[base_m + before_m + __popc(bm & lanemask_lt())] = make_int4(pp.x, pp.y, tp.x, tp.y);
                    acc += sq(b - (double)__ldg(G + tp.x)) + sq(d - (double)__ldg(G + tp.y));
                } else {
                    out[n_m + base_p + before_u + __popc(bu & lanemask_lt())] = make_int4(pp.x, pp.y, -1, -1);
                    acc += 0.5 * sq(d - b);
                }
            }
            base_m += tot_m; base_p += tot_u;
            __syncthreads();
        }
        // G's unmatched intervals, from n_m + n_p
        int base_t = n_m + n_p;
        for (int x0 = 0; x0 < NN; x0 += nt) {
            const int x = x0 + tid;
            const bool u = x < NN && P[1][x] >= 0 && part[1][x] < 0;
            const unsigned bu = __ballot_sync(0xFFFFFFFFu, u);
            if (lane == 0) s_w[0][warp] = __popc(bu);
            __syncthreads();
            int before = 0, tot = 0;
            for (int w = 0; w < kBmThreads / 32; ++w) { const int v = s_w[0][w]; tot += v; if (w < warp) before += v; }
            if (u) {
                const int2 tp = interval_pixels<DIM>(G, H, W, x, (uint32_t)P[1][x]);
                out[base_t + before + __popc(bu & lanemask_lt())] = make_int4(tp.x, tp.y, -1, -1);
                acc += 0.5 * sq((double)__ldg(G + tp.y) - (double)__ldg(G + tp.x));
            }
            base_t += tot;
            __syncthreads();
        }
        if (DIM == 0 && tid == 0) {  // the essential classes: global minimum -> argmax, always matched
            const Geo<0> gl(L, H, W), gg(G, H, W);
            int a, c;
            gl.vertex_val(s_root[0] / gl.VW, s_root[0] % gl.VW, &a);
            gg.vertex_val(s_root[1] / gg.VW, s_root[1] % gg.VW, &c);
            const int ml = (int)(0xFFFFFFFFu - (uint32_t)s_argmax[0]), mg = (int)(0xFFFFFFFFu - (uint32_t)s_argmax[1]);
            out[n_m - 1] = make_int4(a, ml, c, mg);
            acc += sq((double)__ldg(L + a) - (double)__ldg(G + c)) + sq((double)__ldg(L + ml) - (double)__ldg(G + mg));
        }
        acc = block_sum(acc, s_red);
        if (tid == 0) A.cost[map] = (float)acc;
    }
}

// One CTA per map (grid-stride): the map's records, packed by the host-read offsets (int32 [3][n_maps + 1]).
__global__ void __launch_bounds__(256) betti_gather_kernel(const int4* __restrict__ arena, const uint32_t* __restrict__ recoff,
                                                           int n_maps, const int32_t* __restrict__ offsets,
                                                           int2* __restrict__ matched, int2* __restrict__ up, int2* __restrict__ ut) {
    const int32_t* om = offsets;
    const int32_t* op = offsets + (n_maps + 1);
    const int32_t* ot = offsets + 2 * (n_maps + 1);
    for (int map = blockIdx.x; map < n_maps; map += gridDim.x) {
        const int nm = om[map + 1] - om[map], np = op[map + 1] - op[map], ntt = ot[map + 1] - ot[map];
        const int4* recs = arena + recoff[map];
        for (int i = threadIdx.x; i < nm + np + ntt; i += blockDim.x) {
            const int4 r = recs[i];
            if (i < nm) { matched[2 * (om[map] + i)] = make_int2(r.x, r.y); matched[2 * (om[map] + i) + 1] = make_int2(r.z, r.w); }
            else if (i < nm + np) up[op[map] + i - nm] = make_int2(r.x, r.y);
            else ut[ot[map] + i - nm - np] = make_int2(r.x, r.y);
        }
    }
}

struct BettiBwdArgs {
    const float* pred; const float* target;
    int n_maps, N;
    const int32_t* offsets;    // [3][n_maps + 1]
    const int2* matched;       // [M][2] int2 = [M][4]
    const int2* up; const int2* ut;
    const float* grad_cost;    // [n_maps]
    float* grad_pred; float* grad_target;  // grad_target may be null
};

// One CTA per map, as diagram_backward_kernel: zero fill, then the scatter-add of d cost / d value into the critical
// pixels.  Matched: 2 (b_L - b_G) and 2 (d_L - d_G) on the prediction, their negation on the target; unmatched:
// -(d - b) on the creator, (d - b) on the destroyer.  Indices outside the map are skipped.
__global__ void __launch_bounds__(512) betti_backward_kernel(BettiBwdArgs A) {
    const int N = A.N;
    for (int map = blockIdx.x; map < A.n_maps; map += gridDim.x) {
        float* gp = A.grad_pred + (size_t)map * N;
        float* gt = A.grad_target ? A.grad_target + (size_t)map * N : nullptr;
        for (int i = threadIdx.x; i < N; i += blockDim.x) { gp[i] = 0.f; if (gt) gt[i] = 0.f; }
        __syncthreads();  // the fill is visible to the whole CTA before its atomics land on the same lines
        const float* L = A.pred + (size_t)map * N;
        const float* G = A.target + (size_t)map * N;
        const float gc = __ldg(A.grad_cost + map);
        const int32_t* om = A.offsets;
        const int32_t* op = A.offsets + (A.n_maps + 1);
        const int32_t* ot = A.offsets + 2 * (A.n_maps + 1);
        auto ok = [N](int p) { return (unsigned int)p < (unsigned int)N; };
        for (int i = om[map] + threadIdx.x; i < om[map + 1]; i += blockDim.x) {
            const int2 p = A.matched[2 * i], t = A.matched[2 * i + 1];
            if (!(ok(p.x) && ok(p.y) && ok(t.x) && ok(t.y))) continue;
            const float db = 2.f * (__ldg(L + p.x) - __ldg(G + t.x)) * gc, dd = 2.f * (__ldg(L + p.y) - __ldg(G + t.y)) * gc;
            atomicAdd(gp + p.x, db); atomicAdd(gp + p.y, dd);
            if (gt) { atomicAdd(gt + t.x, -db); atomicAdd(gt + t.y, -dd); }
        }
        for (int i = op[map] + threadIdx.x; i < op[map + 1]; i += blockDim.x) {
            const int2 p = A.up[i];
            if (!(ok(p.x) && ok(p.y))) continue;
            const float g = (__ldg(L + p.y) - __ldg(L + p.x)) * gc;
            atomicAdd(gp + p.x, -g); atomicAdd(gp + p.y, g);
        }
        if (gt)
            for (int i = ot[map] + threadIdx.x; i < ot[map + 1]; i += blockDim.x) {
                const int2 p = A.ut[i];
                if (!(ok(p.x) && ok(p.y))) continue;
                const float g = (__ldg(G + p.y) - __ldg(G + p.x)) * gc;
                atomicAdd(gt + p.x, -g); atomicAdd(gt + p.y, g);
            }
        __syncthreads();
    }
}

}  // namespace tl
