// Shared-memory persistence kernel.  One CTA per (image, class) map; maps with more than 65535 nodes
// are processed in BANDS of whole node rows (16-bit node ids local to the band; a 256x256 H1 map is a
// single band); same algorithm as ph_kernel.cuh (elder-linked union-find, then a
// lock-free triplet merge tree), but every latency-critical structure lives in shared memory:
//
//   phase A  level-0 union-find on 16-bit parents        par[65536]            (128 KB)
//   census   basin roots get dense ids in raster order   root mask             (  8 KB)
//            -> per-node basin id written in place into par[], root pixel / root value per basin
//   phase B  triplet table over BASINS only, 16-byte self-contained entries
//            {edge key 64, elder target 32, own root value 32}, updated with ATOMS.CAS.128
//            (reuses phase A's shared memory; K <= ~14.5k basins fit, else global fallback)
//   emit     one pair per basin with a recorded edge and positive persistence
//
// OUTSIDE (H1 only) is node 0xFFFF.  When H*W == 65536 that index is also the last pixel, which is
// sound: the bottom-right pixel's earliest edge is always its bottom boundary edge (largest bitmap
// position among its edges, value = its own), so it merges into OUTSIDE at zero persistence first.
#pragma once
#include "ph_kernel.cuh"
#include "ph_binary.cuh"
#include "match_small.cuh"
#include "grad_kernel.cuh"

namespace tl {

constexpr int kSmallMaxRow = 4097;   // nodes per column (the previous band's last-column labels live in shared memory)
constexpr uint32_t kOut16 = 0xFFFFu;
constexpr uint64_t kRootKey = ~0ull;
constexpr int kParBytes = 65536 * 2;
constexpr int kMaskBytes = 65536 / 8;
constexpr int kSmallSmemBytes = 223 * 1024;  // dynamic shared memory of ph_small_kernel (+ ~3.5 KB static: 227 KB per CTA)

struct __align__(16) TEntry {
    uint64_t ekey;    // key of the edge at which this basin dies (kRootKey: still alive)
    uint32_t target;  // an elder basin it merged into (self while alive)
    uint32_t zval;    // ordered value of this basin's eldest node (immutable)
};

// Triplet table handle: a generic pointer (global fallback) plus the 32-bit shared-window address
// of the same table, computed once, so the hot loops index shared memory without cvta.
struct TRef {
    TEntry* g;
    uint32_t s;
};

template <bool SM>
__device__ __forceinline__ TEntry t_load(const TRef& T, uint32_t x) {
    uint32_t a, b, c, d;
    if (SM) {
        asm volatile("ld.volatile.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(T.s + x * 16u) : "memory");
    } else {
        asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "l"(T.g + x) : "memory");
    }
    TEntry e;
    e.ekey = (uint64_t)a | ((uint64_t)b << 32);
    e.target = c;
    e.zval = d;
    return e;
}

template <bool SM>
__device__ __forceinline__ bool t_cas(const TRef& T, uint32_t x, const TEntry& expect, const TEntry& want) {
    const uint64_t e_hi = (uint64_t)expect.target | ((uint64_t)expect.zval << 32);
    const uint64_t d_hi = (uint64_t)want.target | ((uint64_t)want.zval << 32);
    uint64_t o_lo, o_hi;
    if (SM) {
        asm volatile(
            "{\n .reg .b128 e, d, o;\n mov.b128 e, {%3, %4};\n mov.b128 d, {%5, %6};\n"
            " atom.shared.cas.b128 o, [%2], e, d;\n mov.b128 {%0, %1}, o;\n}\n"
            : "=l"(o_lo), "=l"(o_hi) : "r"(T.s + x * 16u), "l"(expect.ekey), "l"(e_hi), "l"(want.ekey), "l"(d_hi) : "memory");
    } else {
        asm volatile(
            "{\n .reg .b128 e, d, o;\n mov.b128 e, {%3, %4};\n mov.b128 d, {%5, %6};\n"
            " atom.global.cas.b128 o, [%2], e, d;\n mov.b128 {%0, %1}, o;\n}\n"
            : "=l"(o_lo), "=l"(o_hi) : "l"(T.g + x), "l"(expect.ekey), "l"(e_hi), "l"(want.ekey), "l"(d_hi) : "memory");
    }
    return o_lo == expect.ekey && o_hi == e_hi;
}

// elder test between basins (ids are dense in raster order of their root node)
// `rootpix` (root node of every basin) breaks value ties when basin ids are not in raster order of
// their roots (several bands); with a single band the ids themselves are, and rootpix is null.
template <int DIM>
__device__ __forceinline__ bool basin_elder(uint32_t x, uint32_t zx, uint32_t y, uint32_t zy, const uint32_t* rootpix) {
    if (DIM == 1) {
        if (x == 0u) return true;   // OUTSIDE
        if (y == 0u) return false;
    }
    if (zx != zy) return zx < zy;  // (complemented for H1) ordered root values
    const uint32_t px = rootpix ? rootpix[x] : x, py = rootpix ? rootpix[y] : y;
    return DIM == 1 ? px > py : px < py;  // H1: larger raster index = elder; H0: smaller
}


#ifdef TL_STATS
#define TL_STAT(i) (++g_stats_local[i])
__device__ unsigned long long g_stats[8];
#else
#define TL_STAT(i) ((void)0)
#endif
#ifdef TL_STATS
#define TL_SARG , g_stats_local
#define TL_SPARAM , unsigned* g_stats_local
#else
#define TL_SARG
#define TL_SPARAM
#endif

struct __align__(16) CrossEdge {
    uint64_t skey;
    uint32_t la, lb;
};

// one 128-bit store per record (the struct assignment compiles to two 64-bit stores)
__device__ __forceinline__ void store_edge(CrossEdge* p, uint64_t skey, uint32_t la, uint32_t lb) {
    *reinterpret_cast<uint4*>(p) = make_uint4((uint32_t)skey, (uint32_t)(skey >> 32), la, lb);
}
// ... with an L2 eviction policy (TL_OPT_LIST_MODE bit 1)
__device__ __forceinline__ void store_edge_hint(CrossEdge* p, uint64_t skey, uint32_t la, uint32_t lb, uint64_t policy) {
    stg_v4_hint(p, make_uint4((uint32_t)skey, (uint32_t)(skey >> 32), la, lb), policy);
}

// dense edge id -> pixel that gudhi's coface walk reaches from that edge
template <int DIM>
__device__ __forceinline__ int edge_top_eid(const Geo<DIM>& g, uint32_t eid, const FastDiv& divRW) {
    const int RW = 2 * g.W + 1;
    const int i = (int)divRW.div(eid), rem = (int)eid - i * RW;
    return rem < g.W ? g.hedge_top(i, rem) : g.vedge_top(i, rem - g.W);
}

// same for an edge whose VALUE is known (it sits in the table entry): the upper / left pixel is the coface iff it
// attains that value, so ONE map load decides instead of two
template <int DIM>
__device__ __forceinline__ int edge_top_known(const Geo<DIM>& g, uint32_t eid, const FastDiv& divRW, float val) {
    const int RW = 2 * g.W + 1, W = g.W, H = g.H;
    const int i = (int)divRW.div(eid), rem = (int)eid - i * RW;
    if (rem < W) {  // h-edge(i, j) between pixels (i-1, j), (i, j)
        const int j = rem;
        if (i == 0) return j;
        if (i == H) return (H - 1) * W + j;
        return g.px(i - 1, j) == val ? (i - 1) * W + j : i * W + j;
    }
    const int j = rem - W;  // v-edge(i, j) between pixels (i, j-1), (i, j)
    if (j == 0) return i * W;
    if (j == W) return i * W + W - 1;
    return g.px(i, j - 1) == val ? i * W + j - 1 : i * W + j;
}

// ---- packed triplet table: one 64-bit word per basin
//   [ 32-bit ordered edge value | P-bit ordered dense edge id | G-bit target basin ],  P + G <= 32,
// so the whole (value, position) edge key is in the word and every comparison is exact; updated
// with ATOMS.CAS.64.  The basin's own root value sits in a separate array (read at decide time only).
struct Packed {
    uint32_t t_s, z_s;   // shared-window addresses of T64[] and zval[]
    int G;               // bits of the target field
    uint32_t gmask;
};
__device__ __forceinline__ uint64_t pk_load(uint32_t addr) {
    uint64_t v;
    asm volatile("ld.volatile.shared.u64 %0, [%1];" : "=l"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t pk_load32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ bool pk_cas(uint32_t addr, uint64_t expect, uint64_t want) {
    uint64_t old;
    asm volatile("atom.shared.cas.b64 %0, [%1], %2, %3;" : "=l"(old) : "r"(addr), "l"(expect), "l"(want) : "memory");
    return old == expect;
}

__device__ __forceinline__ void cp_async16(uint32_t dst_s, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(dst_s), "l"(src) : "memory");
}
// src_bytes = 0 writes 16 zero bytes (an edge 0-0: a self loop the merge drops at once)
__device__ __forceinline__ void cp_async16_zfill(uint32_t dst_s, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" :: "r"(dst_s), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ uint2 lds_v2(uint32_t addr) {
    uint2 v;
    asm volatile("ld.volatile.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_v2(uint32_t addr, uint2 v) {
    asm volatile("st.volatile.shared.v2.u32 [%0], {%1,%2};" :: "r"(addr), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
    uint16_t v;
    asm volatile("ld.volatile.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr) : "memory");
    return v;
}

#ifndef TL_REFILL_TH
#define TL_REFILL_TH 8
#endif
constexpr int kRefillIdle = TL_REFILL_TH;  // idle lanes that trigger a refill of the warp's edge slots
#ifndef TL_FLAT2
#define TL_FLAT2 1
#endif
#ifndef TL_HOPS
#define TL_HOPS 4   // 3 -> 4: -0.8 % on the C2 step (2 / 5 / 6 / 8: +4.5 / -0.1 / +0.5 / +2.1 %; scripts/gpu_r2j.sh)
#endif
// unroll factors of the fast front end's trip loops (experiments; 1 = as written)
#ifndef TL_UNROLL_L0
#define TL_UNROLL_L0 1
#endif
constexpr int kUnrollL0 = TL_UNROLL_L0;
#ifndef TL_UNROLL_FLATTEN
#define TL_UNROLL_FLATTEN 1
#endif
constexpr int kUnrollFlatten = TL_UNROLL_FLATTEN;
#ifndef TL_UNROLL_CENSUS
#define TL_UNROLL_CENSUS 1
#endif
constexpr int kUnrollCensus = TL_UNROLL_CENSUS;
#ifndef TL_UNROLL_LABEL
#define TL_UNROLL_LABEL 1
#endif
constexpr int kUnrollLabel = TL_UNROLL_LABEL;
#ifndef TL_UNROLL_COMPACT
#define TL_UNROLL_COMPACT 1
#endif
constexpr int kUnrollCompact = TL_UNROLL_COMPACT;
constexpr int kHopsPerIter = TL_HOPS;
constexpr int kRing = 64;  // edges per warp in the shared staging ring (two cp.async batches of 32)

// Lock-free Merge of the warp's slice elist[beg..end) as a warp-synchronous state machine.
// Edges are staged global -> shared with cp.async in coalesced batches of 32 (no register
// scoreboard on the loads) and handed to whichever lanes are idle by ballot rank, so the warp's
// lanes stay equally loaded.  Per iteration every active lane advances BOTH representative walks
// by one hop (two independent 8-byte loads in flight).
template <int DIM>
__device__ __forceinline__ void merge_warpq_packed(const Packed& T, const CrossEdge* __restrict__ elist, int beg, int end,
                                                   uint32_t ring_s, const uint32_t* tie_root TL_SPARAM) {
    const int lane = threadIdx.x & 31;
    const int G = T.G;
    const uint64_t gmask64 = (uint64_t)T.gmask;
    const uint32_t lowmask = (1u << (32 - G)) - 1u;  // the ordered dense edge id fits 32 - G bits
    // The slice is cut into 32 sub-slices of S records, lane l fetches from sub-slice l: a batch of 32 edges
    // is 32 edges that lie S records (tens of pixels) apart, so the edges the warp works on concurrently
    // rarely touch the same basin (neighbouring records almost always do: CAS conflicts).  The last
    // sub-slices are padded with zero records.
    const int real = end - beg;
    const int S = (real + 31) >> 5;
    const int total = S << 5;
    int cons = 0, avail = 0, issued = 0;
    uint32_t x = 0u, y = 0u;
    // sug = [ordered value 32 | ordered edge id | all-ones target]: an entry e (same layout, real target) was recorded
    // at a LATER level than this edge iff e > sug -- one 64-bit compare per hop, no shifts
    uint64_t sug = 0ull, ea = 0ull, eb = 0ull;
    bool active = false, doneA = true, doneB = true;
    // lane l's next record: elist[beg + l * S + batch]; past the lane's real records the copy writes zeros (src-size 0) from
    // any valid address.  One pointer, advanced by a record per batch: the 64-bit index arithmetic is paid once.
    const CrossEdge* lane_src = elist + beg + min(lane * S, max(real - 1, 0));
    int lane_left = max(0, min(S, real - lane * S));  // real records this lane still has to fetch
#define TL_ISSUE()                                                                              \
    do {                                                                                        \
        if (issued < total) cp_async16_zfill(ring_s + (uint32_t)((issued + lane) & (kRing - 1)) * 16u, lane_src, lane_left > 0 ? 16u : 0u); \
        cp_async_commit();                                                                      \
        if (lane_left > 0) { --lane_left; if (lane_left > 0) ++lane_src; }                      \
        issued = min(total, issued + 32);                                                       \
    } while (0)
    if (total > 0) TL_ISSUE();
    if (issued < total) TL_ISSUE();
    for (;;) {
        // refill in batches: hand out new edges only when a quarter of the lanes is idle (or all are),
        // so the ~45-instruction refill section is not paid on every hop
        const unsigned need = __ballot_sync(0xFFFFFFFFu, !active);
        bool any_active = need != 0xFFFFFFFFu;  // warp-uniform
        if ((__popc(need) >= kRefillIdle || need == 0xFFFFFFFFu) && cons < total) {
            const int want = min(__popc(need), total - cons);
            if (cons + want > avail) { cp_async_wait_all(); __syncwarp(); avail = issued; }
            const int take = min(want, avail - cons);
            const int rank = __popc(need & lanemask_lt());
            if (!active && rank < take) {
                const uint32_t a_ = ring_s + (uint32_t)((cons + rank) & (kRing - 1)) * 16u;
                uint32_t k0, k1, la, lb;
                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(k0), "=r"(k1), "=r"(la), "=r"(lb) : "r"(a_) : "memory");
                x = la; y = lb;
                sug = ((uint64_t)k1 << 32) | ((uint64_t)(k0 & lowmask) << G) | gmask64;
                doneA = doneB = false; active = true;
                TL_STAT(1);
            }
            cons += take;
            any_active = any_active || take > 0;
            __syncwarp();  // ring slots read before they may be overwritten
            while (issued < total && issued - cons <= kRing - 32) TL_ISSUE();
        }
        if (!any_active) {
            if (cons >= total) break;
            continue;
        }
        if (active) {
#pragma unroll
            for (int hop = 0; hop < kHopsPerIter; ++hop) {  // several hops per trip through the loop's vote / refill logic
                if (!doneA) { TL_STAT(0); ea = pk_load(T.t_s + x * 8u); }
                if (!doneB) { TL_STAT(0); eb = pk_load(T.t_s + y * 8u); }
                if (!doneA) { if (ea > sug) doneA = true; else x = (uint32_t)ea & T.gmask; }
                if (!doneB) { if (eb > sug) doneB = true; else y = (uint32_t)eb & T.gmask; }
            }
            if (doneA && doneB) {  // (entering this section only once 8 or 16 lanes are ready: +3 % cycles, measured)
                TL_STAT(2);
                if (x == y) {
                    active = false;
                } else {
                    TL_STAT(3);
                    const uint32_t zx = pk_load32(T.z_s + x * 4u), zy = pk_load32(T.z_s + y * 4u);
                    const bool sw = basin_elder<DIM>(y, zy, x, zx, tie_root);
                    const uint32_t xx = sw ? y : x, yy = sw ? x : y;  // yy: the younger representative
                    const uint64_t ey = sw ? ea : eb;
                    if (pk_cas(T.t_s + yy * 8u, ey, (sug & ~gmask64) | xx)) {
                        if ((ey | gmask64) == ~0ull) {
                            active = false;
                        } else {  // re-assert yy's former connection for xx
                            TL_STAT(4);
                            x = xx; y = (uint32_t)ey & T.gmask; sug = ey | gmask64; doneA = doneB = false;
                        }
                    } else {
                        TL_STAT(5);
                        x = xx; y = yy; doneA = doneB = false;
                    }
                }
            }
        }
    }
#undef TL_ISSUE
}

// Lock-free Merge of the edges elist[i..i_end) of this lane, as a state machine executed in lock
// step by the warp.  Per lane: (x, y) are the current nodes of the two walks, doneA/doneB tell
// whether the representative at level skey has been reached (ea / eb hold its entry).
template <int DIM, bool SM>
__device__ __forceinline__ void merge_lanes(const TRef& T, const CrossEdge* __restrict__ elist, int i, int i_end, const uint32_t* tie_root TL_SPARAM) {
    uint32_t x = 0u, y = 0u;
    uint64_t skey = 0ull;
    TEntry ea, eb;
    ea.ekey = eb.ekey = 0ull; ea.target = eb.target = 0u; ea.zval = eb.zval = 0u;
    bool active = false, doneA = true, doneB = true;
    CrossEdge nxt;
    nxt.skey = 0ull; nxt.la = nxt.lb = 0u;
    bool have_next = i < i_end;
    if (have_next) nxt = elist[i];
    for (;;) {
        if (!active && have_next) {
            x = nxt.la; y = nxt.lb; skey = nxt.skey;
            doneA = doneB = false; active = true;
            TL_STAT(1);
            ++i;
            have_next = i < i_end;
            if (have_next) nxt = elist[i];  // prefetch: consumed several iterations from now
        }
        if (!__any_sync(0xFFFFFFFFu, active)) break;
        if (active) {
            if (!doneA) { TL_STAT(0); ea = t_load<SM>(T, x); }
            if (!doneB) { TL_STAT(0); eb = t_load<SM>(T, y); }
            if (!doneA) { if (ea.ekey > skey) doneA = true; else x = ea.target; }
            if (!doneB) { if (eb.ekey > skey) doneB = true; else y = eb.target; }
            if (doneA && doneB) {
                TL_STAT(2);
                if (x == y) {
                    active = false;
                } else {
                    TL_STAT(3);
                    const bool sw = basin_elder<DIM>(y, eb.zval, x, ea.zval, tie_root);
                    const uint32_t xx = sw ? y : x, yy = sw ? x : y;  // yy: the younger representative
                    const TEntry ey = sw ? ea : eb;
                    TEntry want;
                    want.ekey = skey; want.target = xx; want.zval = ey.zval;
                    if (t_cas<SM>(T, yy, ey, want)) {
                        if (ey.ekey == kRootKey) {
                            active = false;
                        } else {  // re-assert yy's former connection for xx
                            TL_STAT(4);
                            x = xx; y = ey.target; skey = ey.ekey; doneA = doneB = false;
                        }
                    } else {
                        TL_STAT(5);
                        x = xx; y = yy; doneA = doneB = false;
                    }
                }
            }
        }
    }
}



// ---- one band of a multi-band map: merge the band's own crossing edges on a packed table in shared memory
//      (band-local basin / edge ids) and move the resulting entries to the map's global 128-bit table; a band
//      whose table does not fit the packed form hands its edges to the cross-band list instead.  Kept out of
//      line: it runs once per band and must not cost the main path registers.
struct BandMergeArgs {
    unsigned char* smem;
    CrossEdge* elist; size_t e_stride; int n_in;
    TEntry* Tg; size_t k_stride; const uint32_t* zvalg;
    int Kb, cid_base, H, W, bw, c0, top_reserved;
    int* n_cross_band;
};

template <int DIM>
__device__ __noinline__ void band_merge(const BandMergeArgs& B TL_SPARAM) {
    const int tid = threadIdx.x, nt = blockDim.x, warp = tid >> 5;
    const int Kb = B.Kb, cid_base = B.cid_base, bw = B.bw, GWb = 2 * B.bw + 1, GW = 2 * B.W + 1, n_in = B.n_in;
    const int n_ids_b = B.H * GWb + bw;
    const int Pb = 32 - __clz(n_ids_b), Gb = 32 - __clz(Kb + 1);
    const size_t ring_b = (size_t)(((Kb + 1) * 8 + 15) & ~15) + (size_t)(((Kb + 1) * 4 + 15) & ~15);
    const bool fits = Pb + Gb <= 32 && ring_b + (size_t)(kPhThreads / 32) * kRing * sizeof(CrossEdge) + (size_t)B.top_reserved <= (size_t)kSmallSmemBytes;
    const uint32_t lowmask_b = (1u << (32 - Gb)) - 1u;
    // band-local dense edge id -> global dense edge id (both order the band's edges like the bitmap does)
    auto pos_global = [&](uint32_t pb) {
        const uint32_t rr = pb / (uint32_t)GWb, rem = pb - rr * (uint32_t)GWb;
        return rem < (uint32_t)bw ? rr * (uint32_t)GW + (uint32_t)B.c0 + rem : rr * (uint32_t)GW + (uint32_t)B.W + (uint32_t)B.c0 + (rem - (uint32_t)bw);
    };
    if (fits) {
        uint64_t* T64b = reinterpret_cast<uint64_t*>(B.smem);
        uint32_t* Z32b = reinterpret_cast<uint32_t*>(B.smem + (((Kb + 1) * 8 + 15) & ~15));
        for (int cc = tid; cc <= Kb; cc += nt) {
            T64b[cc] = (~0ull << Gb) | (uint32_t)cc;
            Z32b[cc] = (cc && (size_t)(cid_base + cc) < B.k_stride) ? B.zvalg[cid_base + cc] : 0u;
        }
        __syncthreads();
        Packed PKb;
        PKb.t_s = (uint32_t)__cvta_generic_to_shared(B.smem);
        PKb.z_s = PKb.t_s + (uint32_t)(((Kb + 1) * 8 + 15) & ~15);
        PKb.G = Gb; PKb.gmask = (1u << Gb) - 1u;
        const int perw = (n_in + (nt >> 5) - 1) / (nt >> 5);
        const int wb = min(n_in, warp * perw), we = min(n_in, wb + perw);
        merge_warpq_packed<DIM>(PKb, B.elist, wb, we, PKb.t_s + (uint32_t)ring_b + (uint32_t)warp * kRing * 16u, nullptr TL_SARG);
        __syncthreads();
        for (int cc = tid + 1; cc <= Kb; cc += nt) {  // global edge ids, global basin ids
            if ((size_t)(cid_base + cc) >= B.k_stride) continue;
            const uint64_t e = T64b[cc];
            const uint64_t up = e >> Gb;
            TEntry out;
            out.zval = Z32b[cc];
            if (up == (~0ull >> Gb)) { out.ekey = kRootKey; out.target = (uint32_t)(cid_base + cc); }
            else {
                const uint32_t idk = (uint32_t)up & lowmask_b;
                const uint32_t pg = pos_global(DIM == 1 ? lowmask_b - idk : idk);
                out.ekey = ((up >> (32 - Gb)) << 32) | (DIM == 1 ? ~pg : pg);
                const uint32_t tl_ = (uint32_t)e & PKb.gmask;
                out.target = tl_ ? (uint32_t)cid_base + tl_ : 0u;
            }
            B.Tg[cid_base + cc] = out;
        }
    } else {
        for (int cc = tid + 1; cc <= Kb; cc += nt) {
            if ((size_t)(cid_base + cc) >= B.k_stride) continue;
            TEntry out;
            out.ekey = kRootKey; out.target = (uint32_t)(cid_base + cc); out.zval = B.zvalg[cid_base + cc];
            B.Tg[cid_base + cc] = out;
        }
        for (int i = tid; i < n_in; i += nt) {
            const uint4 v = __ldcg(reinterpret_cast<const uint4*>(B.elist + i));
            const uint32_t pg = pos_global(DIM == 1 ? ~v.x : v.x);
            const int ix = atomicAdd(B.n_cross_band, 1);
            if ((size_t)ix + (size_t)n_in < B.e_stride)  // the tail never reaches the band's own list: e_stride has a band of slack
                __stcg(reinterpret_cast<uint4*>(B.elist + (B.e_stride - 1 - (size_t)ix)),
                       make_uint4(DIM == 1 ? ~pg : pg, v.y, v.z ? v.z + (uint32_t)cid_base : 0u, v.w ? v.w + (uint32_t)cid_base : 0u));
        }
    }
    __syncthreads();
}

// the gradient job of the launch's tail, out of line so that its registers are not the main path's
constexpr int kGradTilePx = 32768;  // 128 KB of the tail's shared memory
#ifndef TL_GRAD_BULK
#define TL_GRAD_BULK 1
#endif
static_assert(kGradTilePx * 4 + 2 * kGradStageBytes <= kSmallSmemBytes, "tile + two staging buffers must fit the tail's shared memory");
// returns the updated parity bits of the two staging mbarriers (block-uniform)
__device__ __noinline__ unsigned int grad_job(const GradArgs& A, int map, double coef, unsigned char* smem, uint32_t bars_s, unsigned int phase,
                                              unsigned long long* dbg) {
    float* tile = reinterpret_cast<float*>(smem);
    if (A.N <= 4 * kGradTilePx) {  // block-uniform
        if (TL_GRAD_BULK) return grad_one_map_tiled_bulk(A, map, coef, 1.0, tile, kGradTilePx, smem + kGradTilePx * 4, bars_s, phase, dbg);
        grad_one_map_tiled(A, map, coef, 1.0, tile, kGradTilePx, dbg);
    } else grad_one_map(A, map, coef, 1.0);
    return phase;
}

struct PhSmallArgs {
    PhArgs base;
    CrossEdge* elist;    // [grid][e_stride] edges that cross two basins
    size_t e_stride;
    uint32_t* rootpix;   // [grid][k_stride] root node of each basin
    uint32_t* zval;      // [grid][k_stride]
    TEntry* T2g;         // [grid][k_stride] fallback triplet table
    size_t k_stride;
    unsigned long long* prof;  // optional [8] phase cycle counters
    int binary_path;           // 1: try the two-valued fast path first (H1)
    int list_mode;             // TL_OPT_LIST_MODE: L2 treatment of the crossing-edge list (single-band maps)
    // tl_forward only: the SM that completes a map's second diagram writes the map's cost itself when one of the two
    // diagrams is empty (ready[k] = 4), else hands the map (ready[k] = 3) to the CTAs that have run out of persistence
    // jobs: the matching runs in the tail of this launch instead of a launch of its own
    int fuse_match;
    unsigned int* ready;       // [n_maps] sets of map k that are finished (device counters, zeroed by the host)
    MatchFwdArgs mf;
    // tl_forward_backward only: the same tail also writes the gradient (upstream 1.0) of every image whose C maps are
    // matched.  An image is PUBLISHED by the CTA that matches its last map: gq[slot] = kGqValid | image (| kGqSkip when
    // one of its maps went to the heavy list: tl_backward's grad_kernel serves those); its C maps are C gradient jobs,
    // claimed in publication order from gq_head -- only jobs whose image is already published, so nobody waits while holding one.
    int fuse_grad;
    GradArgs ga;               // coef / grad_loss unused: the coefficient is formed from `cost` per job
    const double* cost;        // [n_maps] matching cost per map (MatchFwdArgs::cost)
    unsigned int* img_cnt;     // [B] low 16 bits: matched maps of the image, high 16: of those, maps on the heavy list
    unsigned int* gq;          // [B] publication queue
    unsigned int* gq_tail;     // images published
    unsigned int* gq_head;     // gradient jobs claimed
    uint32_t* gfused;          // [B] 1: the image's gradient has been written here
};
constexpr unsigned int kGqValid = 0x80000000u, kGqSkip = 0x40000000u, kGqImage = 0x00FFFFFFu;

template <int DIM>
struct SmallCtx {
    Geo<DIM> g;
    uint16_t* par;
    // the band: columns c0 .. c0+bw-1 of every row; ids in par[] are local, r * bw + (c - c0)
    int bw, c0, rowlen;
    FastDiv divB;
    __device__ __forceinline__ SmallCtx(const float* f, int H, int W, uint16_t* par_) : g(f, H, W), par(par_), bw(1), c0(0), rowlen(1), divB(1u) {}
    __device__ __forceinline__ int glob(uint32_t xl) const { const int r = (int)divB.div(xl); return r * rowlen + c0 + (int)xl - r * bw; }

    __device__ __forceinline__ uint32_t find(uint32_t x) const {
        volatile uint16_t* p = par;
        uint32_t px = p[x];
        while (px != x) {
            const uint32_t gp = p[px];
            if (gp != px) p[x] = (uint16_t)gp;  // path halving; non-root entries only ever hold ancestors
            x = px; px = gp;
        }
        return x;
    }
    // read-only find for the flatten pass: a halving store there could land after another thread
    // has already flattened that entry and regress it to a non-root ancestor
    __device__ __forceinline__ uint32_t find_ro(uint32_t x) const {
        const volatile uint16_t* p = par;
        uint32_t px = p[x];
        while (px != x) { x = px; px = p[x]; }
        return x;
    }
    __device__ __forceinline__ bool elder(uint32_t x, uint32_t y) const {
        if (DIM == 1) {
            if (x == kOut16) return true;
            if (y == kOut16) return false;
        }
        return g.nkey(glob(x)) < g.nkey(glob(y));
    }
    __device__ void union0(uint32_t a, uint32_t b) {
        for (;;) {
            uint32_t ra = find(a), rb = find(b);
            if (ra == rb) return;
            if (elder(rb, ra)) { uint32_t t = ra; ra = rb; rb = t; }
            const unsigned short old = atomicCAS(reinterpret_cast<unsigned short*>(par + rb), (unsigned short)rb, (unsigned short)ra);
            if (old == (unsigned short)rb) return;
            a = ra; b = rb;
        }
    }
};

// MULTI = false: the host guarantees a single band (<= 65536 pixels / <= 65535 vertices): the band loop runs
// once and everything that serves band borders is compiled out of the headline kernel.
template <int DIM, bool MULTI>
__global__ void __launch_bounds__(kPhThreads, 1) ph_small_kernel(const __grid_constant__ PhSmallArgs S) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ unsigned int s_job, s_next;
    __shared__ int s_count, s_K, s_ncross, s_nan, s_nx;
    __shared__ unsigned long long s_argmax;
    __shared__ unsigned int s_lo, s_hi;
    __shared__ int s_wcnt[kPhThreads / 32];
    __shared__ double s_red[kPhThreads / 32];
    __shared__ unsigned long long s_base;
    const PhArgs& A = S.base;
    // (single-band kernel only: TL_OPT_LIST_MODE bit 2 reads the maps without the evict-last hint, bit 1 stores the list with it)
    const bool list_keep = !MULTI && (S.list_mode & 2) != 0;
    const uint64_t l2_last = l2_policy_evict_last();
    const uint64_t l2_keep = (!MULTI && (S.list_mode & 4)) ? l2_policy_evict_normal() : l2_last;
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const int H = A.H, W = A.W, N = H * W;
    uint16_t* par = reinterpret_cast<uint16_t*>(smem);
    uint32_t* mask = reinterpret_cast<uint32_t*>(smem + kParBytes);
    TEntry* Ts = reinterpret_cast<TEntry*>(smem);
    const int t_cap_smem = kSmallSmemBytes / (int)sizeof(TEntry);
    uint32_t* rootpix = S.rootpix + (size_t)blockIdx.x * S.k_stride;
    uint32_t* zvalg = S.zval + (size_t)blockIdx.x * S.k_stride;
    const unsigned int n_jobs = (unsigned)A.n_sets * (unsigned)A.n_maps;
    long long t0 = 0;
#ifdef TL_STATS
    unsigned g_stats_local[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif
#define TL_PROF(slot)                                                        \
    do {                                                                     \
        if (S.prof && tid == 0) { long long t1 = clock64(); atomicAdd(S.prof + (slot), (unsigned long long)(t1 - t0)); t0 = t1; } \
    } while (0)

    if (tid == 0) s_next = atomicAdd(A.job_counter, 1u);
    int finished_map = -1;  // (thread 0) map of the job just completed, to be published
    // (thread 0, tl_forward_backward) map k has its final cost -- or sits on the heavy list: count it for its image and,
    // when it is the image's last map, publish the image to the gradient queue
    auto map_matched = [&](int k, bool heavy) {
        __threadfence();
        const unsigned int b = (unsigned int)(k / S.ga.C);
        const unsigned int old = atomicAdd(S.img_cnt + b, heavy ? 0x10001u : 1u);
        if ((old & 0xFFFFu) + 1u == (unsigned int)S.ga.C) {
            const bool skip = (old >> 16) != 0u || heavy;
            if (!skip) S.gfused[b] = 1u;
            const unsigned int slot = atomicAdd(S.gq_tail, 1u);
            __threadfence();
            asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(S.gq + slot), "r"(kGqValid | (skip ? kGqSkip : 0u) | b) : "memory");
        }
    };
    for (;;) {
        __syncthreads();
        // publish the finished job: every thread's records are written (barrier above), release them device-wide.
        // ready[k]: 0 / 1 / 2 = finished diagrams of map k; the SM that finishes the second one then sets 3 = "both
        // complete, to be matched by a job of the tail" or -- when one of the diagrams is empty, most maps with
        // segmentation ground truth: the cost is the two diagonal sums -- writes the cost itself and sets 4 = "matched"
        if (tid == 0 && finished_map >= 0 && S.fuse_match) {
            __threadfence();
            if (atomicAdd(S.ready + finished_map, 1u) == 1u) {
                unsigned int st = 3u;
                if (!S.mf.loss_r) {
                    __threadfence();
                    const int n0 = __ldcg(A.ps.counts[0] + finished_map), n1 = __ldcg(A.ps.counts[1] + finished_map);
                    if (n0 == 0 || n1 == 0) {
                        S.mf.cost[finished_map] = __ldcg(A.ps.dsum[0] + finished_map) + __ldcg(A.ps.dsum[1] + finished_map);
                        S.mf.tpers[finished_map] = 0.0;
                        st = 4u;
                        if (S.fuse_grad) map_matched(finished_map, false);
                    }
                }
                __threadfence();
                asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(S.ready + finished_map), "r"(st) : "memory");
            }
        }
        // one job is always claimed ahead: its map is prefetched into L2 while this one is being emitted
        if (tid == 0) { s_job = s_next; s_next = atomicAdd(A.job_counter, 1u); s_count = 0; s_ncross = 0; s_nx = 0; s_nan = 0; s_argmax = 0ull; s_lo = 0xFFFFFFFFu; s_hi = 0u; }
        __syncthreads();
        const unsigned int job = s_job;
        if (job >= n_jobs) break;
        if (S.prof && tid == 0) t0 = clock64();
        // all prediction maps first (heavy), ground-truth maps (light) fill the tail of the launch
        const int set = (int)(job / (unsigned)A.n_maps), map = (int)(job % (unsigned)A.n_maps);
        finished_map = map;
        // two-valued maps (one-hot ground truth): run-based labelling on a bit mask, no merge tree; a probe of
        // the first words sends every other map on to the generic path
        if (DIM == 1 && S.binary_path &&
            binary_h1_pairs(A.maps[set] + (size_t)map * N, H, W, smem, kSmallSmemBytes, A.ps, set, map, S.prof)) {
            TL_PROF(0);
            continue;
        }
        SmallCtx<DIM> cx(A.maps[set] + (size_t)map * N, H, W, par);
        const Geo<DIM>& g = cx.g;
        const int NN = g.NN, GW = g.GW, VW = g.VW;

        // fast front end (H1, one band, rows of whole 128-bit quads): phases 0-3 and the compaction run
        // on 4 consecutive pixels per lane, see below; every other shape takes the generic banded path
        // (maps with more than 65535 pixels go through it in bands of whole columns, 4-column aligned)
        const bool fast = DIM == 1 && (W & 3) == 0 && H <= 16383 && (reinterpret_cast<uintptr_t>(g.f) & 15) == 0;
        const bool fast_one = fast && N <= 65536;  // single band: min / max fused into level 0

        // ---- phase 0: init, argmax (H0), and the constant-map shortcut (absent classes give all-zero
        //      ground-truth maps: no finite pair; H0 keeps only the essential class (0 -> argmax = 0))
        if (!fast_one) {
            unsigned long long best = 0ull;
            uint32_t lo = 0xFFFFFFFFu, hi = 0u;
            bool has_nan = false;
            if ((N & 3) == 0 && (reinterpret_cast<uintptr_t>(g.f) & 15) == 0) {
                const float4* f4 = reinterpret_cast<const float4*>(g.f);
#pragma unroll 4
                for (int q = tid; q < (N >> 2); q += nt) {  // coalesced 128-bit loads
                    const float4 v = __ldg(f4 + q);
                    const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t m = mono32(vv[k]);
                        has_nan |= vv[k] != vv[k];
                        lo = min(lo, m); hi = max(hi, m);
                        if (DIM == 0) {
                            unsigned long long kk = ((unsigned long long)m << 32) | (uint32_t)(0xFFFFFFFFu - (uint32_t)(4 * q + k));
                            best = kk > best ? kk : best;
                        }
                    }
                }
            } else {
#pragma unroll 4
                for (int p = tid; p < N; p += nt) {
                    const float fv = __ldg(g.f + p);
                    const uint32_t m = mono32(fv);
                    has_nan |= fv != fv;
                    lo = min(lo, m); hi = max(hi, m);
                    if (DIM == 0) {
                        unsigned long long k = ((unsigned long long)m << 32) | (uint32_t)(0xFFFFFFFFu - (uint32_t)p);
                        best = k > best ? k : best;
                    }
                }
            }
            lo = __reduce_min_sync(0xFFFFFFFFu, lo); hi = __reduce_max_sync(0xFFFFFFFFu, hi);
            if (lane == 0) { atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
            if (DIM == 0) atomicMax(&s_argmax, best);
            if (has_nan) s_nan = 1;
        }
        __syncthreads();
        if (!fast_one) TL_PROF(0);
        if (!fast_one && s_nan) {  // block-uniform: the (value, position) order is undefined with a NaN
            if (tid == 0) { int av; atomicOr(A.ps.status, kStNonFinite); ps_reserve(A.ps, set, map, 0, &av); A.ps.dsum[set][map] = 0.0; }
            continue;
        }
        if (!fast_one && s_lo == s_hi) {  // block-uniform
            if (tid == 0) {
                int avail;
                const unsigned long long base = ps_reserve(A.ps, set, map, DIM == 0 ? 1 : 0, &avail);
                double ds = 0.0;
                if (DIM == 0 && avail > 0) {  // H0 keeps only the essential class (0 -> argmax = 0)
                    PairRec rec;
                    rec.cre = 0; rec.des = 0; rec.b = rec.d = __ldg(g.f);
                    rec.tb = rec.td = __int_as_float(0x7FC00000);
                    A.ps.arena[base] = rec;
                    if (A.ps.skeys) A.ps.skeys[base] = ~0ull;
                    ds = (double)cost_diag(rec.b, rec.d, A.ps.q);
                }
                A.ps.dsum[set][map] = ds;
            }
            continue;
        }

        // ---- phases 1-3 run per BAND of whole node COLUMNS (<= 65535 nodes, 16-bit ids local to the
        //      band; a 256x256 H1 map is one band).  Level-0 links never leave a band: a node whose
        //      earliest edge crosses the band border stays the root of its sub-basin and that edge is
        //      handed to the merge tree as an ordinary crossing edge.  Still exact: forest paths stay
        //      key-monotone, a sub-basin root is the eldest node of its sub-basin, and the deferred merge
        //      has zero persistence (tests/test_algorithm_model.py runs the banded variant too).
        //      Column bands because ties resolve vertically first (H1: the edge below is the earliest of
        //      equal edges, H0: the edge above), so plateaus contract inside a band instead of leaving one
        //      sub-basin per column.
        const int rowlen = DIM == 1 ? W : VW, n_rows = DIM == 1 ? H : H + 1;
        const int n_rows_all = n_rows;
        const bool alias = DIM == 1 && N == 65536;  // single band whose last pixel doubles as OUTSIDE
        const int cols_per_band = alias ? rowlen : fast ? min(rowlen, (65535 / n_rows) & ~3) : min(rowlen, 65535 / n_rows);
        const bool one_band = !MULTI || cols_per_band >= rowlen;
        // labels of the previous band's last column: at the top of shared memory, out of the way of the in-band table
        uint32_t* prev_lab = reinterpret_cast<uint32_t*>(smem + kSmallSmemBytes - 4 * (size_t)(n_rows_all));
        CrossEdge* elist = S.elist + (size_t)blockIdx.x * S.e_stride;
        int cid_base = 0;  // basins found in earlier bands
        // pick(r, c): step (dr, dc) to the far end of node (r,c)'s earliest incident edge when that edge
        // has the node's own value; out = the far end is OUTSIDE; none = strict local extremum (stays a
        // root); elder_far = the far end is known to be ELDER than the node from registers alone
        auto pick = [&](int r, int c, int& dr, int& dc, bool& out, bool& none, bool& elder_far) {
            dr = dc = 0; out = false; none = false; elder_far = false;
            const int x = r * rowlen + c;
            if (DIM == 1) {
                const float fp = g.px(r, c);
                const float fu = r == 0 ? fp : g.px(r - 1, c), fd = r == H - 1 ? fp : g.px(r + 1, c);
                const float fl = c == 0 ? fp : g.px(r, c - 1), fr = c == W - 1 ? fp : g.px(r, c + 1);
                // earliest incident edge in the descending scan = largest (value, position): the
                // value is fp whenever the far pixel is >= fp (or the edge is a boundary edge), and
                // among those the bitmap position orders bottom > right > left > top
                float fo = fp;
                if (r == H - 1) out = true;
                else if (fd >= fp) { dr = 1; fo = fd; }
                else if (c == W - 1) out = true;
                else if (fr >= fp) { dc = 1; fo = fr; }
                else if (c == 0) out = true;
                else if (fl >= fp) { dc = -1; fo = fl; }
                else if (r == 0) out = true;
                else if (fu >= fp) { dr = -1; fo = fu; }
                else none = true;  // strict local maximum
                // strictly higher, OUTSIDE, or equal with a larger raster index: elder than the node
                elder_far = out || fo > fp || (fo == fp && (dr > 0 || dc > 0));
                if (alias && !out && !none && x + dr * rowlen + dc == N - 1) { out = true; elder_far = true; }
            } else {
                uint64_t best = ~0ull;
                if (r > 0) {
                    uint64_t k = g.make_ekey(g.vedge_val(r - 1, c), (uint32_t)(2 * c + (2 * r - 1) * GW));
                    if (k < best) { best = k; dr = -1; dc = 0; }
                }
                if (r < H) {
                    uint64_t k = g.make_ekey(g.vedge_val(r, c), (uint32_t)(2 * c + (2 * r + 1) * GW));
                    if (k < best) { best = k; dr = 1; dc = 0; }
                }
                if (c > 0) {
                    uint64_t k = g.make_ekey(g.hedge_val(r, c - 1), (uint32_t)(2 * c - 1 + (2 * r) * GW));
                    if (k < best) { best = k; dr = 0; dc = -1; }
                }
                if (c < W) {
                    uint64_t k = g.make_ekey(g.hedge_val(r, c), (uint32_t)(2 * c + 1 + (2 * r) * GW));
                    if (k < best) { best = k; dr = 0; dc = 1; }
                }
                // a vertex always has an incident edge of its own value: never `none`.  The far vertex is a
                // face of that edge, so its value is <= the edge's = the node's own: it is elder when it
                // comes earlier in raster order (up / left), or when its value is strictly smaller
                if (dr < 0 || dc < 0) elder_far = true;
                else elder_far = mono32(g.vertex_val(r + dr, c + dc, nullptr)) < (uint32_t)(best >> 32);
            }
        };
        // Maps of several bands (fast front end): every band's own crossing edges are merged right away on a
        // packed table in SHARED memory (band-local basin and edge ids), the resulting entries are written to
        // the map's global table, and only the edges that cross a band border (one per row and border) are
        // left for the final merge on that global table.  Exact for the same reason the merge accepts edges
        // in any order: entries are facts, and a band's facts stay true in the whole map.
        const bool inband = MULTI && fast && !one_band;
        if (fast) {
            // ================= fast front end =================
            // Every warp owns a contiguous chunk of whole 128-node groups; per trip a lane owns the 4
            // consecutive pixels x .. x+3 of one row (W % 4 == 0), so the map is read with 128-bit loads
            // (own row, row above, row below + the two scalars left / right of the quad) and par[] is
            // read and written 4 entries (8 bytes) at a time.  The same ownership is kept through
            // level 0, flatten, census and labelling, so root flags stay in registers.
            // Maps with more than 65535 pixels are processed in bands of whole columns (a multiple of 4
            // wide): ids in par[] are band-local, r * bw + (c - c0); level-0 links never leave a band (a
            // pixel whose earliest edge crosses the band border stays the root of its sub-basin and the
            // deferred zero-persistence merge goes to the merge tree), see the generic path below.
            const float* __restrict__ f = g.f;
            for (int c0 = 0; c0 < W; c0 += cols_per_band) {
            const int c1 = min(W, c0 + cols_per_band), bw = c1 - c0, nb = H * bw;  // this band: columns c0 .. c1-1
            const FastDiv divW = bw == W ? FastDiv(A.magic_W, (uint32_t)W) : FastDiv((uint32_t)bw);
            const int chunk = ((nb + 32 * 128 - 1) / (32 * 128)) * 128;  // nodes per warp
            const int wbeg = min(nb, warp * chunk), wend = min(nb, wbeg + chunk);
            const int trips = (wend - wbeg + 127) >> 7;                  // <= 16
            cx.bw = bw; cx.c0 = c0; cx.rowlen = W; cx.divB = divW;
            __syncthreads();  // the previous band's readers of par[] are done
            if (tid == 0) { par[kOut16] = (uint16_t)kOut16; if (inband) s_ncross = 0; }  // OUTSIDE's own entry (alias: the last pixel)
            // ---- level 0a: pick pointers, min / max of the map, tie flags for level 0b
            {
                float vlo = __int_as_float(0x7F800000), vhi = __int_as_float(0xFF800000);
                bool nan_seen = false;
#pragma unroll kUnrollL0
                for (int t = 0; t < trips; ++t) {
                    const int x = wbeg + t * 128 + lane * 4;  // band-local id of the quad
                    unsigned defer = 0u;
                    if (x < wend) {
                        const int r = (int)divW.div((uint32_t)x), cl = x - r * bw, c = c0 + cl;
                        const float* q = f + r * W + c;
                        const float4 M = ldg_f4_keep(reinterpret_cast<const float4*>(q), l2_keep);
                        const float4 U = r > 0 ? ldg_f4_keep(reinterpret_cast<const float4*>(q - W), l2_keep) : M;
                        const float4 D = r < H - 1 ? ldg_f4_keep(reinterpret_cast<const float4*>(q + W), l2_keep) : M;
                        const float L = c > 0 ? __ldg(q - 1) : 0.f;
                        const float R = c + 4 < W ? __ldg(q + 4) : 0.f;
                        vlo = fminf(vlo, fminf(fminf(M.x, M.y), fminf(M.z, M.w)));
                        vhi = fmaxf(vhi, fmaxf(fmaxf(M.x, M.y), fmaxf(M.z, M.w)));
                        nan_seen |= (M.x != M.x) | (M.y != M.y) | (M.z != M.z) | (M.w != M.w);
                        const float m[6] = {L, M.x, M.y, M.z, M.w, R};
                        const float u[4] = {U.x, U.y, U.z, U.w}, d[4] = {D.x, D.y, D.z, D.w};
                        uint32_t pk[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            // earliest incident edge of the descending scan among the edges that carry the
                            // pixel's own value: bottom > right > left > top by bitmap position; a far end that
                            // is higher, OUTSIDE, or equal with a larger raster index is elder: plain pointer;
                            // a far end in another band: no link (the pixel stays a sub-basin root)
                            const float fp = m[k + 1];
                            const int xk = x + k;
                            uint32_t tgt = (uint32_t)xk;
                            bool direct = true;
                            if (r == H - 1) tgt = kOut16;
                            else if (d[k] >= fp) tgt = (uint32_t)(xk + bw);
                            else if (c + k == W - 1) tgt = kOut16;
                            else if (m[k + 2] >= fp) { if (cl + k + 1 < bw) tgt = (uint32_t)(xk + 1); }
                            else if (c + k == 0) tgt = kOut16;
                            else if (m[k] >= fp) { if (cl + k > 0) { tgt = (uint32_t)(xk - 1); direct = m[k] > fp; } }
                            else if (r == 0) tgt = kOut16;
                            else if (u[k] >= fp) { tgt = (uint32_t)(xk - bw); direct = u[k] > fp; }
                            if (alias && xk == N - 1) { tgt = kOut16; direct = true; }  // the pixel that doubles as OUTSIDE keeps itself
                            if (!direct) { defer |= 1u << k; tgt = (uint32_t)xk; }
                            pk[k] = tgt;
                        }
                        *reinterpret_cast<uint2*>(par + x) = make_uint2(pk[0] | (pk[1] << 16), pk[2] | (pk[3] << 16));
                    }
                    // tie flags in node order: 4 words per trip
                    if (wbeg + t * 128 < wend) {
                        const unsigned any = __ballot_sync(0xFFFFFFFFu, defer != 0u);
                        unsigned v = 0u;
                        if (any) {
                            v = defer << (4 * (lane & 7));
                            v |= __shfl_xor_sync(0xFFFFFFFFu, v, 1);
                            v |= __shfl_xor_sync(0xFFFFFFFFu, v, 2);
                            v |= __shfl_xor_sync(0xFFFFFFFFu, v, 4);
                        }
                        if ((lane & 7) == 0) mask[((wbeg + t * 128) >> 5) + (lane >> 3)] = v;
                    }
                }
                // constant-map shortcut (absent classes give all-zero ground-truth maps: no finite pair);
                // banded maps took it in phase 0
                if (fast_one) {
                    if (nan_seen) s_nan = 1;
                    const uint32_t lo = __reduce_min_sync(0xFFFFFFFFu, mono32(vlo)), hi = __reduce_max_sync(0xFFFFFFFFu, mono32(vhi));
                    if (lane == 0 && wbeg < wend) { atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
                }
            }
            __syncthreads();
            if (fast_one && (s_lo == s_hi || s_nan)) break;  // block-uniform: constant / NaN map, handled after the band loop
            // ---- level 0b: elder-linked lock-free unions for the tie-flagged nodes
            for (int w0 = warp; w0 < ((nb + 31) >> 5); w0 += nt >> 5) {
                const unsigned bits = mask[w0];
                if (bits) {
                    const int xl = w0 * 32 + lane;
                    if ((bits >> lane) & 1u) {
                        const int r = (int)divW.div((uint32_t)xl), c = c0 + xl - r * bw;
                        int dr, dc; bool out, none, ef;
                        pick(r, c, dr, dc, out, none, ef);
                        if (!none && (out || (c + dc >= c0 && c + dc < c1)))
                            cx.union0((uint32_t)xl, out ? kOut16 : (uint32_t)(xl + dr * bw + dc));
                    }
                    __syncwarp();
                }
            }
            __syncthreads();
            TL_PROF(1);
            // ---- flatten by pointer jumping, 4 own entries per trip; a node is finished once its parent
            //      is a root (roots are final after level 0), finished quads are skipped
            unsigned long long rootbits = 0ull, donebits = 0ull;
            const uint32_t par_s = (uint32_t)__cvta_generic_to_shared(par);
            for (int round = 0;; ++round) {
                int pending = 0;
                // bottom rows first: most ties point DOWN (plateaus), so a row that jumps after the rows below it
                // sees their already shortened pointers and a vertical run collapses within one round
#pragma unroll kUnrollFlatten
                for (int t = trips - 1; t >= 0; --t) {
                    const int x = wbeg + t * 128 + lane * 4;
                    const bool act = x < wend && ((donebits >> (4 * t)) & 15ull) != 15ull;
                    if (!__any_sync(0xFFFFFFFFu, act)) continue;
                    if (act) {
                        const uint2 w = lds_v2(par_s + 2u * (uint32_t)x);
                        const uint32_t p0 = w.x & 0xFFFFu, p1 = w.x >> 16, p2 = w.y & 0xFFFFu, p3 = w.y >> 16;
#if TL_FLAT2
                        // two jumps per round (parent's parent's parent): a third fewer block-wide rounds on the long
                        // pointer chains of plateaus
                        const uint32_t q0 = lds_u16(par_s + 2u * p0), q1 = lds_u16(par_s + 2u * p1), q2 = lds_u16(par_s + 2u * p2), q3 = lds_u16(par_s + 2u * p3);
                        const uint32_t g0 = lds_u16(par_s + 2u * q0), g1 = lds_u16(par_s + 2u * q1), g2 = lds_u16(par_s + 2u * q2), g3 = lds_u16(par_s + 2u * q3);
#else
                        const uint32_t g0 = lds_u16(par_s + 2u * p0), g1 = lds_u16(par_s + 2u * p1), g2 = lds_u16(par_s + 2u * p2), g3 = lds_u16(par_s + 2u * p3);
                        const uint32_t q0 = p0, q1 = p1, q2 = p2, q3 = p3;
#endif
                        if (round == 0) {
                            const unsigned rb = (p0 == (uint32_t)x ? 1u : 0u) | (p1 == (uint32_t)x + 1u ? 2u : 0u) |
                                                (p2 == (uint32_t)x + 2u ? 4u : 0u) | (p3 == (uint32_t)x + 3u ? 8u : 0u);
                            rootbits |= (unsigned long long)rb << (4 * t);
                        }
                        const unsigned dn = (g0 == q0 ? 1u : 0u) | (g1 == q1 ? 2u : 0u) | (g2 == q2 ? 4u : 0u) | (g3 == q3 ? 8u : 0u);
                        donebits |= (unsigned long long)dn << (4 * t);
                        if (g0 != p0 || g1 != p1 || g2 != p2 || g3 != p3)
                            sts_v2(par_s + 2u * (uint32_t)x, make_uint2(g0 | (g1 << 16), g2 | (g3 << 16)));
                        if (dn != 15u) pending = 1;
                    }
                }
                if (!__syncthreads_or(pending)) break;
            }
            if (alias && wend == N && lane == 31) rootbits &= ~(8ull << (4 * (trips - 1)));  // node N-1 is OUTSIDE, not a basin
            TL_PROF(2);
            // ---- census: dense basin ids in (band-local) raster order of the roots
            {
                const int cnt = __reduce_add_sync(0xFFFFFFFFu, __popcll(rootbits));
                if (lane == 0) s_wcnt[warp] = cnt;
            }
            __syncthreads();
            if (warp == 0) {
                const int v = s_wcnt[lane];
                int incl = v;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
                s_wcnt[lane] = incl - v;
                if (lane == 31) s_K = incl;
            }
            __syncthreads();
            const int Kb = s_K;  // basins of this band: global ids cid_base+1 .. cid_base+Kb
            {
                int run = s_wcnt[warp];
#pragma unroll kUnrollCensus
                for (int t = 0; t < trips; ++t) {
                    const int x = wbeg + t * 128 + lane * 4;
                    const unsigned nib = (unsigned)(rootbits >> (4 * t)) & 15u;
                    const int c = __popc(nib);
                    int incl = c;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += v; }
                    if (nib) {
                        uint2 w = *reinterpret_cast<const uint2*>(par + x);
                        int rank = run + incl - c;  // 0-based inside the band
                        const int r = (int)divW.div((uint32_t)x), gx = r * W + c0 + x - r * bw;  // global pixel of the quad
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            if ((nib >> k) & 1u) {
                                // (a single band's tables hold the combinatorial maximum, and its root values are read
                                // from the map when the table is set up: all lanes busy there, a fifth of them here)
                                if (!MULTI) rootpix[rank + 1] = (uint32_t)(gx + k);
                                else if (cid_base + rank + 1 < (int)S.k_stride) {
                                    rootpix[cid_base + rank + 1] = (uint32_t)(gx + k);
                                    zvalg[cid_base + rank + 1] = ~mono32(__ldg(f + gx + k));
                                }
                                // the root's entry becomes its LABEL: band-local rank + 1 (0 will stand for OUTSIDE)
                                ++rank;
                                if (k == 0) w.x = (w.x & 0xFFFF0000u) | (uint32_t)rank;
                                else if (k == 1) w.x = (w.x & 0x0000FFFFu) | ((uint32_t)rank << 16);
                                else if (k == 2) w.y = (w.y & 0xFFFF0000u) | (uint32_t)rank;
                                else w.y = (w.y & 0x0000FFFFu) | ((uint32_t)rank << 16);
                            }
                        }
                        *reinterpret_cast<uint2*>(par + x) = w;
                    }
                    run += __shfl_sync(0xFFFFFFFFu, incl, 31);
                }
            }
            __syncthreads();
            if (tid == 0) par[kOut16] = 0;  // OUTSIDE's label (its own barrier: with the alias the entry sits in a quad the census may rewrite)
            __syncthreads();
            // per-node label in place: band-local basin rank + 1, 0 for OUTSIDE's basin.  Root entries are labels already;
            // every other entry holds its root's index, or kOut16, whose entry is OUTSIDE's label: one load, no test
#pragma unroll kUnrollLabel
            for (int t = 0; t < trips; ++t) {
                const int x = wbeg + t * 128 + lane * 4;
                unsigned nib = (unsigned)(rootbits >> (4 * t)) & 15u;
                if (alias && x + 3 == N - 1) nib |= 8u;  // the pixel that doubles as OUTSIDE: its entry IS OUTSIDE's label, just set
                if (x < wend && nib != 15u) {
                    const uint2 w = *reinterpret_cast<const uint2*>(par + x);
                    uint32_t e[4] = {w.x & 0xFFFFu, w.x >> 16, w.y & 0xFFFFu, w.y >> 16};
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (!((nib >> k) & 1u)) e[k] = par[e[k]];
                    *reinterpret_cast<uint2*>(par + x) = make_uint2(e[0] | (e[1] << 16), e[2] | (e[3] << 16));
                }
            }
            __syncthreads();
            TL_PROF(3);
            // ---- compaction: the edges that cross two basins go to the per-CTA list.  Every pixel owns the
            //      v-edge to its left and the h-edge above it (the left edge of a band's first column reaches
            //      into the previous band, whose last-column labels are kept in prev_lab); the last column /
            //      row also own the boundary edges to OUTSIDE.  Dense edge ids as in the generic path.
            // Labels and dense edge ids are BAND-LOCAL (basin rank + 1, 0 = OUTSIDE; bitmap row pair i of the band
            // holds its bw h-edges, then its bw + 1 v-edges): with a single band that is the global numbering.
            // Only the left edge of a band's first column leaves the band: it goes, with global labels and a
            // global edge id, to the cross-band list that grows down from the end of the CTA's list.
            auto glab = [&](uint32_t v) { return v ? (uint32_t)cid_base + v : 0u; };  // band-local label -> map-wide label
            auto llab = [&](uint32_t v) { return v; };
            const int GWb = 2 * bw + 1;
#pragma unroll kUnrollCompact
            for (int t = 0; t < trips; ++t) {  // warp-uniform trip count
                const int x = wbeg + t * 128 + lane * 4;
                const bool valid = x < wend;
                unsigned flags = 0u;
                uint32_t lab[5] = {0u, 0u, 0u, 0u, 0u}, ulab[4] = {0u, 0u, 0u, 0u};  // lab[0]: left of the quad
                float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f}, u[4] = {0.f, 0.f, 0.f, 0.f};
                int r = 0, c = 0, cl = 0;
                bool xband = false;  // the quad's left edge crosses into the previous band
                if (valid) {
                    r = (int)divW.div((uint32_t)x);
                    cl = x - r * bw;
                    c = c0 + cl;
                    xband = MULTI && cl == 0 && c > 0;
                    const uint2 w = *reinterpret_cast<const uint2*>(par + x);
                    lab[1] = llab(w.x & 0xFFFFu); lab[2] = llab(w.x >> 16); lab[3] = llab(w.y & 0xFFFFu); lab[4] = llab(w.y >> 16);
                    if (cl > 0) lab[0] = llab(par[x - 1]);
                    if (r > 0) {
                        const uint2 wu = *reinterpret_cast<const uint2*>(par + x - bw);
                        ulab[0] = llab(wu.x & 0xFFFFu); ulab[1] = llab(wu.x >> 16); ulab[2] = llab(wu.y & 0xFFFFu); ulab[3] = llab(wu.y >> 16);
                    }
                    const float* q = f + r * W + c;
                    const float4 M = ldg_f4_keep(reinterpret_cast<const float4*>(q), l2_keep);
                    m[1] = M.x; m[2] = M.y; m[3] = M.z; m[4] = M.w;
                    if (c > 0) m[0] = __ldg(q - 1);
                    if (r > 0) {
                        const float4 U = ldg_f4_keep(reinterpret_cast<const float4*>(q - W), l2_keep);
                        u[0] = U.x; u[1] = U.y; u[2] = U.z; u[3] = U.w;
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint32_t own = lab[k + 1];
                        if (lab[k] != own && !(k == 0 && xband)) flags |= 1u << (4 * k);  // left v-edge (boundary edge when c + k == 0)
                        if (ulab[k] != own) flags |= 2u << (4 * k);     // top h-edge (boundary edge when r == 0)
                        if (c + k == W - 1 && own != 0u) flags |= 4u << (4 * k);
                        if (r == H - 1 && own != 0u) flags |= 8u << (4 * k);
                    }
                    // Same-pair duplicates that are visible in registers: of two crossing edges that join the SAME two
                    // basins only the earlier one (larger value, then larger position) can be a tree edge.
                    //  (i)  a pixel's left and top edge lead into the same basin;
                    //  (ii) the top edges of two neighbouring pixels of one basin lead into the same basin.
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const unsigned lf = 1u << (4 * k), tp = 2u << (4 * k);
                        if ((flags & lf) && (flags & tp) && lab[k] == ulab[k]) {
                            const float vl = c + k == 0 ? m[k + 1] : fminf(m[k], m[k + 1]), vt = r == 0 ? m[k + 1] : fminf(u[k], m[k + 1]);
                            flags &= vt > vl ? ~lf : ~tp;  // on a tie the v-edge (larger position) is the earlier one
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        const unsigned t0 = 2u << (4 * k), t1 = 2u << (4 * (k + 1));
                        if ((flags & t0) && (flags & t1) && lab[k + 1] == lab[k + 2] && ulab[k] == ulab[k + 1]) {
                            const float v0 = r == 0 ? m[k + 1] : fminf(u[k], m[k + 1]), v1 = r == 0 ? m[k + 2] : fminf(u[k + 1], m[k + 2]);
                            flags &= v0 > v1 ? ~t1 : ~t0;  // on a tie the right-hand edge (larger position) is the earlier one
                        }
                    }
                    if (xband) {  // always crossing: level-0 links never leave a band
                        const int ix = atomicAdd(&s_nx, 1);
                        const uint32_t posg = (uint32_t)(r * GW + W + c);
                        if (ix < (int)S.e_stride) store_edge(elist + (S.e_stride - 1 - (size_t)ix), g.make_ekey(fminf(m[0], m[1]), posg), prev_lab[r], glab(w.x & 0xFFFFu));
                    }
                }
                const int cnt = __popc(flags);
                int incl = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += v; }
                int slot = 0;
                if (lane == 31 && incl > 0) slot = atomicAdd(&s_ncross, incl);
                slot = __shfl_sync(0xFFFFFFFFu, slot, 31) + incl - cnt;
                if (flags) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const float fp = m[k + 1];
                        const uint32_t own = lab[k + 1];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            if (flags & (1u << (4 * k + e))) {
                                uint32_t lo, pos;
                                float val;
                                if (e == 0) { lo = lab[k]; pos = (uint32_t)(r * GWb + bw + cl + k); val = c + k == 0 ? fp : fminf(m[k], fp); }
                                else if (e == 1) { lo = ulab[k]; pos = (uint32_t)(r * GWb + cl + k); val = r == 0 ? fp : fminf(u[k], fp); }
                                else if (e == 2) { lo = 0u; pos = (uint32_t)(r * GWb + 2 * bw); val = fp; }
                                else { lo = 0u; pos = (uint32_t)(H * GWb + cl + k); val = fp; }
                                if (slot < (int)S.e_stride) {
                                    if (list_keep) store_edge_hint(elist + slot, g.make_ekey(val, pos), lo, own, l2_last);
                                    else store_edge(elist + slot, g.make_ekey(val, pos), lo, own);
                                }
                                ++slot;
                            }
                        }
                    }
                }
            }
            __syncthreads();
            // labels of this band's last column, for the next band's "left" edges
            if (c1 < W)
                for (int r = tid; r < H; r += nt) prev_lab[r] = glab(par[r * bw + bw - 1]);
            TL_PROF(6);
            if (inband) {
                __syncthreads();  // prev_lab is written and every label has been read: the band's table may take the space
                BandMergeArgs bm;
                bm.smem = smem; bm.elist = elist; bm.e_stride = S.e_stride; bm.n_in = min(s_ncross, (int)S.e_stride);
                bm.Tg = S.T2g + (size_t)blockIdx.x * S.k_stride; bm.k_stride = S.k_stride; bm.zvalg = zvalg;
                bm.Kb = Kb; bm.cid_base = cid_base; bm.H = H; bm.W = W; bm.bw = bw; bm.c0 = c0; bm.top_reserved = 4 * n_rows_all;
                bm.n_cross_band = &s_nx;
                band_merge<DIM>(bm TL_SARG);
                TL_PROF(4);
            }
            cid_base += Kb;
            }  // bands
            if (fast_one && (s_lo == s_hi || s_nan)) {  // block-uniform: constant map, or a NaN pixel (pairing undefined)
                if (tid == 0) { int avail; if (s_nan) atomicOr(A.ps.status, kStNonFinite); ps_reserve(A.ps, set, map, 0, &avail); A.ps.dsum[set][map] = 0.0; }
                TL_PROF(0);
                continue;
            }
        } else
        for (int c0 = 0; c0 < rowlen; c0 += cols_per_band) {
            const int c1 = min(rowlen, c0 + cols_per_band), bw = c1 - c0, nb = n_rows * bw;  // this band: columns c0 .. c1-1
            const FastDiv divB((uint32_t)bw);
            cx.bw = bw; cx.c0 = c0; cx.rowlen = rowlen; cx.divB = divB;
            // far end of a pick as a band-local id: kOut16 for OUTSIDE, -1 when it lies outside the band
            // (then no level-0 link is made) or when the node is a strict extremum
            auto far_local = [&](int xl, int c, int dr, int dc, bool out, bool none) {
                if (none) return -1;
                if (out) return (int)kOut16;
                const int c2 = c + dc;
                return (c2 < c0 || c2 >= c1) ? -1 : xl + dr * bw + dc;
            };
            __syncthreads();
            for (int x = tid; x < 65536; x += nt) par[x] = (uint16_t)x;
            __syncthreads();
            // phase 1a: a node whose far end is elder by registers just POINTS at it -- a plain store to
            // its own entry, no atomics, no find (every entry has one writer in this phase).  The others
            // (ties towards a smaller raster index; every H0 vertex) are flagged for phase 1b.
            // 4 nodes per lane per trip so that the 4 x 5 map loads are in flight together.
            for (int x0 = warp * 32; x0 < nb; x0 += 4 * nt) {  // warp-uniform trip count
                int other[4];
                bool elder_far[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int xl = x0 + u * nt + lane;
                    other[u] = -1; elder_far[u] = false;
                    if (xl < nb && !(alias && xl == N - 1)) {
                        const int r = (int)divB.div((uint32_t)xl), c = c0 + xl - r * bw;
                        int dr, dc; bool out, none;
                        pick(r, c, dr, dc, out, none, elder_far[u]);
                        other[u] = far_local(xl, c, dr, dc, out, none);
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int xl = x0 + u * nt + lane;
                    const bool direct = other[u] >= 0 && elder_far[u];
                    if (direct) par[xl] = (uint16_t)other[u];
                    const unsigned deferred = __ballot_sync(0xFFFFFFFFu, other[u] >= 0 && !direct);
                    if (lane == 0 && x0 + u * nt < nb) mask[(x0 + u * nt) >> 5] = deferred;
                }
            }
            __syncthreads();
            // phase 1b: elder-linked lock-free unions (CAS on the younger root) for the flagged nodes
            for (int w0 = warp; w0 < ((nb + 31) >> 5); w0 += nt >> 5) {
                const unsigned bits = mask[w0];
                if (bits) {
                    const int xl = w0 * 32 + lane;
                    if ((bits >> lane) & 1u) {
                        const int r = (int)divB.div((uint32_t)xl), c = c0 + xl - r * bw;
                        int dr, dc; bool out, none, ef;
                        pick(r, c, dr, dc, out, none, ef);
                        const int oth = far_local(xl, c, dr, dc, out, none);
                        if (oth >= 0) cx.union0((uint32_t)xl, (uint32_t)oth);
                    }
                    __syncwarp();  // reconverge: without it the lanes drift apart and replay the loop body per group
                }
            }
            __syncthreads();
            TL_PROF(1);
            // flatten by pointer jumping: each round every node adopts its grandparent (own entry only,
            // so no store can regress another thread's result); depth halves per round
            for (;;) {
                int changed = 0;
#pragma unroll 4
                for (int x = tid; x < nb; x += nt) {
                    const uint32_t p = par[x];
                    const uint32_t gp = par[p];
                    if (gp != p) { par[x] = (uint16_t)gp; changed = 1; }
                }
                if (!__syncthreads_or(changed)) break;
            }
            TL_PROF(2);

            // ---- census: dense basin ids in band-local raster order of the roots (with a single band
            //      that is the global raster order, which then serves as the tie-break between basins)
            const int chunk = (((nb + 31) / 32) + 31) & ~31;
            const int beg = min(nb, warp * chunk), end = min(nb, beg + chunk);
            {
                int cnt = 0;
                for (int i0 = beg; i0 < end; i0 += 32) {
                    const int i = i0 + lane;
                    const bool root = i < end && par[i] == (uint16_t)i && !(DIM == 1 && (uint32_t)i == kOut16);
                    cnt += __popc(__ballot_sync(0xFFFFFFFFu, root));
                }
                if (lane == 0) s_wcnt[warp] = cnt;
            }
            __syncthreads();
            if (warp == 0) {
                const int v = s_wcnt[lane];
                int incl = v;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
                s_wcnt[lane] = incl - v;
                if (lane == 31) s_K = incl;
            }
            __syncthreads();
            const int Kb = s_K;  // basins of this band: global ids cid_base+1 .. cid_base+Kb
            {
                int run = s_wcnt[warp];
                for (int i0 = beg; i0 < end; i0 += 32) {
                    const int i = i0 + lane;
                    const bool root = i < end && par[i] == (uint16_t)i && !(DIM == 1 && (uint32_t)i == kOut16);
                    const unsigned bal = __ballot_sync(0xFFFFFFFFu, root);
                    if (lane == 0) mask[i0 >> 5] = bal;
                    if (root) {
                        const int rank = run + __popc(bal & lanemask_lt());  // 0-based inside the band
                        const int gx = cx.glob((uint32_t)i);
                        if (cid_base + 1 + rank < (int)S.k_stride) {
                            rootpix[cid_base + 1 + rank] = (uint32_t)gx;
                            zvalg[cid_base + 1 + rank] = (uint32_t)(g.nkey(gx) >> 32);
                        }
                        par[i] = (uint16_t)rank;
                    }
                    run += __popc(bal);
                }
            }
            __syncthreads();
            // per-node label in place: band-local basin rank, kOut16 for OUTSIDE's basin
#pragma unroll 4
            for (int x = tid; x < nb; x += nt) {
                uint32_t b;
                if ((mask[x >> 5] >> (x & 31)) & 1u) b = par[x];
                else {
                    const uint32_t r = par[x];
                    b = (DIM == 1 && r == kOut16) ? kOut16 : par[r];
                }
                par[x] = (uint16_t)b;  // after the flatten nobody reads a non-root entry, roots keep their rank
            }
            __syncthreads();
            TL_PROF(3);

            // ---- compaction: the edges that cross two basins go to a per-CTA list.  Every node owns the
            //      edge to its left and the edge above it (H1: pixel; H0: vertex), so only the "left" edge
            //      can cross into the previous band, whose last-column labels are kept in prev_lab; H1's
            //      last column / row also own the boundary edges to OUTSIDE.  `pos` below is the DENSE edge
            //      id: rank of the edge among edges in bitmap order (bitmap row pair i holds W h-edges then
            //      W+1 v-edges), order-isomorphic to the bitmap position.  2 nodes per lane per trip.
            auto glabel = [&](uint32_t v) { return v == kOut16 ? 0u : (uint32_t)(cid_base + 1) + v; };
            for (int x0 = warp * 32; x0 < nb; x0 += 2 * nt) {  // warp-uniform trip count
                uint32_t lab[2], lo1[2], lo2[2];
                int rr[2], cc[2];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int xl = x0 + u * nt + lane;
                    lab[u] = lo1[u] = lo2[u] = 0u; rr[u] = cc[u] = 0;
                    if (xl < nb) {
                        rr[u] = (int)divB.div((uint32_t)xl); cc[u] = c0 + xl - rr[u] * bw;
                        lab[u] = glabel(par[xl]);
                        const bool first_col = cc[u] == c0;
                        if (DIM == 1) {
                            lo1[u] = cc[u] == 0 ? 0u : first_col ? prev_lab[rr[u]] : glabel(par[xl - 1]);  // left v-edge
                            lo2[u] = rr[u] == 0 ? 0u : glabel(par[xl - bw]);                                // top h-edge
                        } else {
                            lo1[u] = rr[u] == 0 ? lab[u] : glabel(par[xl - bw]);                            // up v-edge
                            lo2[u] = cc[u] == 0 ? lab[u] : first_col ? prev_lab[rr[u]] : glabel(par[xl - 1]);  // left h-edge
                        }
                    }
                }
                // count this lane's crossing edges (at most 8 flags), ONE warp scan + ONE atomic per trip,
                // then form and store the records
                unsigned flags = 0u;
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int xl = x0 + u * nt + lane;
                    if (xl < nb) {
                        if (lo1[u] != lab[u]) flags |= 1u << (4 * u);
                        if (lo2[u] != lab[u]) flags |= 2u << (4 * u);
                        if (DIM == 1) {
                            if (cc[u] == W - 1 && lab[u] != 0u) flags |= 4u << (4 * u);
                            if (rr[u] == H - 1 && lab[u] != 0u) flags |= 8u << (4 * u);
                        }
                    }
                }
                const int cnt = __popc(flags);
                int incl = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
                int slot = 0;
                if (lane == 31 && incl > 0) slot = atomicAdd(&s_ncross, incl);
                slot = __shfl_sync(0xFFFFFFFFu, slot, 31) + incl - cnt;
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int r = rr[u], c = cc[u];
#pragma unroll
                    for (int k = 0; k < (DIM == 1 ? 4 : 2); ++k) {
                        // k = 0 / 1: the two owned edges; k = 2 / 3: right / bottom boundary edges (H1 only)
                        if (flags & (1u << (4 * u + k))) {
                            uint32_t lo = 0u, pos;
                            float val;
                            if (DIM == 1) {
                                if (k == 0) { lo = lo1[u]; pos = (uint32_t)(r * GW + W + c); val = g.vedge_val(r, c); }
                                else if (k == 1) { lo = lo2[u]; pos = (uint32_t)(r * GW + c); val = g.hedge_val(r, c); }
                                else if (k == 2) { pos = (uint32_t)(r * GW + 2 * W); val = g.px(r, c); }
                                else { pos = (uint32_t)(H * GW + c); val = g.px(r, c); }
                            } else {
                                // vertex (r,c): up v-edge(r-1,c) joins (r-1,c),(r,c); left h-edge(r,c-1) joins (r,c-1),(r,c)
                                if (k == 0) { lo = lo1[u]; pos = (uint32_t)((r - 1) * GW + W + c); val = g.vedge_val(r - 1, c); }
                                else { lo = lo2[u]; pos = (uint32_t)(r * GW + c - 1); val = g.hedge_val(r, c - 1); }
                            }
                            if (slot < (int)S.e_stride) store_edge(elist + slot, g.make_ekey(val, pos), lo, lab[u]);
                            ++slot;
                        }
                    }
                }
            }
            __syncthreads();
            // labels of this band's last column, for the next band's "left" edges
            if (c1 < rowlen)
                for (int r = tid; r < n_rows; r += nt) prev_lab[r] = glabel(par[r * bw + bw - 1]);
            cid_base += Kb;
            TL_PROF(6);
        }
        const int K = cid_base;  // basins 1..K (0 = OUTSIDE for H1, unused for H0)
        if ((size_t)K + 2 > S.k_stride) {  // block-uniform; only with the typical-size tables of multi-band maps
            if (tid == 0) { int av; atomicOr(A.ps.status, kStBasins); ps_reserve(A.ps, set, map, 0, &av); A.ps.dsum[set][map] = 0.0; }
            continue;
        }

        // ---- phase B: triplet merge tree over basins
        // packed 64-bit entries when edge id + basin id fit 32 bits next to the 32-bit value (always
        // exact); otherwise 128-bit entries, in shared memory if they fit, else in the global spill
        const int n_edge_ids = H * GW + W;  // dense ids 0 .. H*(2W+1)+W-1
        const int Pbits = 32 - __clz(n_edge_ids), Gbits = 32 - __clz(K + 1);
        const size_t ring_off = (size_t)(((K + 1) * 8 + 15) & ~15) + (size_t)(((K + 1) * 4 + 15) & ~15);
        // (maps merged band by band already hold their entries in the global table: 128-bit form, global memory)
        const bool packed = !inband && Pbits + Gbits <= 32 && ring_off + (size_t)(kPhThreads / 32) * kRing * sizeof(CrossEdge) <= (size_t)kSmallSmemBytes;
        const bool t_in_smem = !inband && K + 1 <= t_cap_smem;
        TRef T;
        T.g = t_in_smem ? Ts : S.T2g + (size_t)blockIdx.x * S.k_stride;
        T.s = (uint32_t)__cvta_generic_to_shared(Ts);
        Packed PK;
        PK.t_s = T.s; PK.z_s = T.s + (uint32_t)(((K + 1) * 8 + 15) & ~15); PK.G = Gbits; PK.gmask = (1u << Gbits) - 1u;
        uint64_t* T64 = reinterpret_cast<uint64_t*>(smem);
        uint32_t* Z32 = reinterpret_cast<uint32_t*>(smem + (((K + 1) * 8 + 15) & ~15));
        __syncthreads();  // every basin id has been read: the union-find storage can become the table
        // emission scratch in shared memory (packed case): the compact list of emitting basins borrows the
        // staging ring after the merge; the root pixel of every basin sits behind the ring when it fits
        // (16-bit when node ids do), so the emission's dependent global loads shrink to the map values
        const size_t rp_off = ring_off + (size_t)(kPhThreads / 32) * kRing * sizeof(CrossEdge);
        const bool rp16 = (DIM == 1 ? N : NN) <= 65536;  // root node ids fit 16 bits
        const bool rp_smem = packed && rp_off + (size_t)(K + 1) * (rp16 ? 2 : 4) <= (size_t)kSmallSmemBytes;
        const bool lst_smem = packed && (size_t)K * 2 <= (size_t)(kPhThreads / 32) * kRing * sizeof(CrossEdge);
        uint16_t* rp_s16 = reinterpret_cast<uint16_t*>(smem + rp_off);
        uint32_t* rp_s32 = reinterpret_cast<uint32_t*>(smem + rp_off);
        uint16_t* lst16 = reinterpret_cast<uint16_t*>(smem + ring_off);
        // root value of basin c: the fast front end of a single-band map left it in the map (see the census)
        const bool z_in_map = fast && !MULTI;
        auto zval_of = [&](int c, uint32_t rp) { return z_in_map ? ~mono32(__ldg(g.f + rp)) : zvalg[c]; };
        if (packed) {
#pragma unroll 4
            for (int c = tid; c <= K; c += nt) {  // (unrolled: root pixel, then its value, are dependent loads from L2)
                const uint32_t rp = c && (rp_smem || z_in_map) ? rootpix[c] : 0u;
                T64[c] = (~0ull << Gbits) | (uint32_t)c; Z32[c] = c ? zval_of(c, rp) : 0u;
                if (rp_smem) { if (rp16) rp_s16[c] = (uint16_t)rp; else rp_s32[c] = rp; }
            }
        } else if (inband) {
            if (tid == 0) { TEntry e; e.ekey = kRootKey; e.target = 0u; e.zval = 0u; T.g[0] = e; }  // OUTSIDE; the bands wrote the rest
        } else {
            for (int c = tid; c <= K; c += nt) {
                TEntry e;
                e.ekey = kRootKey; e.target = (uint32_t)c; e.zval = c ? zval_of(c, z_in_map ? rootpix[c] : 0u) : 0u;
                T.g[c] = e;
            }
        }
        __syncthreads();
        TL_PROF(6);  // phase 4a: crossing-edge compaction + table init
        // pass 2: every lane owns a contiguous chunk of the list (all lanes have work; concurrently
        // processed edges are far apart -> few CAS conflicts).  The merge is a warp-synchronous state
        // machine: per iteration every active lane advances BOTH representative walks by one hop (two
        // independent 16-byte loads in flight), so lanes stay converged instead of serialising
        // differently long walks.
        {
            // in-band mode: what is left are the edges across band borders, at the END of the CTA's list
            const int n_cross = inband ? min(s_nx, (int)S.e_stride) : min(s_ncross, (int)S.e_stride);
            if (inband) elist += S.e_stride - (size_t)n_cross;
            const uint32_t* tie_root = one_band ? nullptr : rootpix;
            if (packed) {  // contiguous slice per warp, edges handed to idle lanes
                const int perw = (n_cross + (nt >> 5) - 1) / (nt >> 5);
                const int wb = min(n_cross, warp * perw), we = min(n_cross, wb + perw);
                merge_warpq_packed<DIM>(PK, elist, wb, we, T.s + (uint32_t)ring_off + (uint32_t)warp * kRing * 16u, tie_root TL_SARG);
            } else {       // contiguous chunk per lane
                const int per = (n_cross + nt - 1) / nt;
                int i = min(n_cross, tid * per);
                const int i_end = min(n_cross, i + per);
                if (t_in_smem) merge_lanes<DIM, true>(T, elist, i, i_end, tie_root TL_SARG);
                else merge_lanes<DIM, false>(T, elist, i, i_end, tie_root TL_SARG);
            }
        }
#ifdef TL_STATS
        for (int i = 0; i < 8; ++i) if (g_stats_local[i]) { atomicAdd(&g_stats[i], (unsigned long long)g_stats_local[i]); g_stats_local[i] = 0; }
        if (tid == 0) { atomicAdd(&g_stats[6], (unsigned long long)K); atomicAdd(&g_stats[7], 1ull); }
#endif
        __syncthreads();
        // the list has been consumed and is scratch: let L2 drop its lines instead of writing them back (TL_OPT_LIST_MODE
        // bit 0).  Whole 128-byte lines of this CTA's own slot only (slots are multiples of 1 KB)
        if (!MULTI && (S.list_mode & 1)) {
            const int n_lines = (min(s_ncross, (int)S.e_stride) * (int)sizeof(CrossEdge) + 127) >> 7;
            const char* lb_ = reinterpret_cast<const char*>(elist);
            if ((reinterpret_cast<uintptr_t>(lb_) & 127) == 0)
                for (int i = tid; i < n_lines; i += nt) l2_discard_line(lb_ + (size_t)i * 128);
        }
        TL_PROF(4);

        // ---- emit: every thread owns a contiguous run of basins, so ONE block scan yields
        //      deterministic slots in basin (= raster) order
        const FastDiv divRW(A.magic_GW, (uint32_t)GW), divVW(A.magic_VW, (uint32_t)VW);  // exact for ids < 2^24 (multiply-shift)
        {   // the next job's map: one 128-byte line per prefetch, into L2 only (it is read once)
            const unsigned int nj = s_next;
            if (nj < n_jobs) {
                const char* nm = reinterpret_cast<const char*>(A.maps[nj / (unsigned)A.n_maps] + (size_t)(nj % (unsigned)A.n_maps) * N);
                for (int i = tid; i < (N * 4 + 127) / 128; i += nt) asm volatile("prefetch.global.L2 [%0];" :: "l"(nm + (size_t)i * 128));
            }
        }
        {
            auto load_entry = [&](int c, uint64_t& ekey, uint32_t& zv) {
                if (packed) {
                    const uint64_t up = T64[c] >> Gbits;  // [value 32 | ordered edge id]
                    zv = Z32[c];
                    if (up == (~0ull >> Gbits)) { ekey = kRootKey; return; }
                    const uint32_t lowmask = (1u << (32 - Gbits)) - 1u;
                    const uint32_t idk = (uint32_t)up & lowmask;
                    // restore the full-width ordered id (complemented for H1) used by the 128-bit form
                    ekey = ((up >> (32 - Gbits)) << 32) | (DIM == 1 ? ~(lowmask - idk) : idk);
                } else {
                    const TEntry e = t_in_smem ? t_load<true>(T, (uint32_t)c) : t_load<false>(T, (uint32_t)c);
                    ekey = e.ekey; zv = e.zval;
                }
            };
            // rounds of up to 64 contiguous basins per thread (one 64-bit flag word); each round: flags,
            // one block scan, append the emitting basin ids to the compact list (zvalg is free after the
            // table was initialised)
            const int per = min(64, (K + nt - 1) / nt);
            int total = 0;
            for (int c_round = 1; c_round <= K; c_round += per * nt) {
                const int c_beg = c_round + tid * per, c_end = min(K + 1, c_beg + per);
                unsigned long long flags = 0ull;
                for (int c = c_beg; c < c_end; ++c) {
                    uint64_t ekey; uint32_t zv;
                    load_entry(c, ekey, zv);
                    const bool emit = ekey != kRootKey ? (uint32_t)(ekey >> 32) != zv : DIM == 0;  // essential class (H0)
                    if (emit) flags |= 1ull << (c - c_beg);
                }
                const int cnt = __popcll(flags);
                int incl = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= o) incl += t; }
                __syncthreads();  // previous round's readers of s_wcnt are done
                if (lane == 31) s_wcnt[warp] = incl;
                __syncthreads();
                int slot = total + incl - cnt;
                for (int w = 0; w < kPhThreads / 32; ++w) { const int v = s_wcnt[w]; total += v; if (w < warp) slot += v; }
                for (int c = c_beg; c < c_end; ++c)
                    if ((flags >> (c - c_beg)) & 1ull) { if (lst_smem) lst16[slot] = (uint16_t)c; else zvalg[slot] = (uint32_t)c; ++slot; }
            }
            // the map's records: one reservation in the shared arena
            if (tid == 0) { int av; s_base = ps_reserve(A.ps, set, map, total, &av); s_count = av; }
            __syncthreads();
            PairRec* out = A.ps.arena + s_base;
            uint64_t* skeys = A.ps.skeys ? A.ps.skeys + s_base : nullptr;
            const int avail = s_count;
            double dacc = 0.0;  // sum of the points' costs to the diagonal (the matching kernel's column term)
            // 4 records per thread per trip, staged so that the global loads of the 4 records overlap; per
            // record the only dependent global accesses are the two map values that decide the edge's pixel
            for (int j0 = tid; j0 < total; j0 += 4 * nt) {
                int cc4[4], xx4[4];
                uint64_t ek4[4];
                uint32_t zv4[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) { const int j = j0 + u * nt; cc4[u] = j < total ? (lst_smem ? (int)lst16[j] : (int)zvalg[j]) : 0; }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int j = j0 + u * nt;
                    xx4[u] = 0; ek4[u] = kRootKey; zv4[u] = 0u;
                    if (j < total) {
                        xx4[u] = rp_smem ? (rp16 ? (int)rp_s16[cc4[u]] : (int)rp_s32[cc4[u]]) : (int)rootpix[cc4[u]];
                        load_entry(cc4[u], ek4[u], zv4[u]);
                    }
                }
                PairRec rec4[4];
                uint64_t sk4[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int j = j0 + u * nt;
                    rec4[u].cre = rec4[u].des = 0; rec4[u].b = rec4[u].d = 0.f; sk4[u] = 0ull;
                    if (j >= total) continue;
                    const int x = xx4[u];
                    if (ek4[u] == kRootKey) {  // H0 essential class: paired with argmax, emitted last by gudhi
                        { const int vi = (int)divVW.div((uint32_t)x); rec4[u].b = g.vertex_val(vi, x - vi * VW, &rec4[u].cre); }
                        rec4[u].des = (int)(0xFFFFFFFFu - (uint32_t)s_argmax);
                        rec4[u].d = __ldg(g.f + rec4[u].des);
                        sk4[u] = ~0ull;
                    } else if (DIM == 1) {
                        // birth / death values come out of the table (exact inverse of the ordered keys): the only
                        // map access left is the one load that tells which pixel of the edge attains its value
                        rec4[u].des = x;
                        rec4[u].d = unmono32(~zv4[u]);
                        rec4[u].b = unmono32(~(uint32_t)(ek4[u] >> 32));
                        rec4[u].cre = edge_top_known<DIM>(g, (uint32_t)(~ek4[u]), divRW, rec4[u].b);
                        sk4[u] = ((uint64_t)(~zv4[u]) << 32) | (uint32_t)x;  // death cell = square x
                    } else {
                        { const int vi = (int)divVW.div((uint32_t)x); rec4[u].b = g.vertex_val(vi, x - vi * VW, &rec4[u].cre); }
                        rec4[u].d = unmono32((uint32_t)(ek4[u] >> 32));
                        rec4[u].des = edge_top_known<DIM>(g, (uint32_t)ek4[u], divRW, rec4[u].d);
                        sk4[u] = ek4[u];  // death cell = edge
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int j = j0 + u * nt;
                    if (j < avail) {
                        rec4[u].tb = rec4[u].td = __int_as_float(0x7FC00000);
                        {   // written once, read by later kernels only: stream past L2
                            const uint2* rw = reinterpret_cast<const uint2*>(&rec4[u]);
                            uint2* ow = reinterpret_cast<uint2*>(out + j);
                            __stcs(ow, rw[0]); __stcs(ow + 1, rw[1]); __stcs(ow + 2, rw[2]);
                        }
                        if (skeys) skeys[j] = sk4[u];
                        dacc += (double)cost_diag(rec4[u].b, rec4[u].d, A.ps.q);
                    }
                }
            }
            dacc = block_sum(dacc, s_red);
            if (tid == 0) A.ps.dsum[set][map] = dacc;
        }
        TL_PROF(5);
    }
    // ---- tail of the launch: this SM has no persistence job left.  Match the maps whose prediction and ground-truth
    //      diagrams are both complete (the other SMs are still finishing theirs) and, for tl_forward_backward, write
    //      the gradient of the images whose maps are all matched.  Thread 0 is the scheduler.  Jobs of both kinds are
    //      claimed with a fetch-add (a compare-and-swap claim serialises the 148 SMs on one word: measured 0.4 ms), so
    //      a claimed job may not be runnable yet (matching: ready[k] < 3; gradient: image not published): the SM keeps
    //      at most one job of each kind in hand and runs whichever becomes runnable first.  No cycle of waits: a held
    //      gradient job waits for matching jobs, which wait for persistence jobs, which wait for nothing, and an SM
    //      holding a gradient job keeps claiming and running matching jobs.  The next job of a kind is claimed right
    //      before the current one runs, so the claim's round trip to L2 hides behind the job.
    // TL_OPT_PROFILE: per-CTA timeline of the tail (ns, %globaltimer) in the CTA's own root-pixel scratch, free by now:
    // [0] persistence jobs done  [1] exit  [2] ns in matching jobs  [3] ns in gradient jobs  [4] matching jobs  [5] gradient jobs
    unsigned long long tp_t0 = 0ull, tp_match = 0ull, tp_grad = 0ull, tp_nm = 0ull, tp_ng = 0ull;
    auto now_ns = [] { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; };
    if (S.prof && tid == 0) tp_t0 = now_ns();
    __shared__ unsigned long long s_gdbg[5];
    if (tid == 0) s_gdbg[0] = s_gdbg[1] = s_gdbg[2] = s_gdbg[3] = s_gdbg[4] = 0ull;
    if (S.fuse_match) {
        __shared__ int s_kind, s_arg;
        __shared__ double s_coef;
        __shared__ __align__(8) unsigned long long s_bars[2];  // completion barriers of the gradient jobs' record stream
        const uint32_t bars_s = (uint32_t)__cvta_generic_to_shared(s_bars);
        unsigned int bar_phase = 0u;
        if (tid == 0) { mbar_init(bars_s, 1u); mbar_init(bars_s + 8u, 1u); mbar_init_fence(); }
        const int n_maps = S.mf.n_maps, Cc = S.ga.C;
        const unsigned int n_gjobs = S.fuse_grad ? (unsigned int)n_maps : 0u;
        // (thread 0) claimed job of each kind: kNoJob = none in hand, >= limit = that kind is exhausted
        constexpr unsigned int kNoJob = 0xFFFFFFFFu;
        unsigned int held_m = kNoJob, held_g = kNoJob;
        bool m_done = false, g_done = n_gjobs == 0u;
        if (tid == 0) {
            held_m = atomicAdd(S.mf.counter, 1u);
            if (!g_done) held_g = atomicAdd(S.gq_head, 1u);
        }
        for (;;) {
            __syncthreads();
            if (tid == 0) {
                int kind = 0, arg = 0;
                for (;;) {
                    if (!m_done && held_m == kNoJob) held_m = atomicAdd(S.mf.counter, 1u);
                    if (!g_done && held_g == kNoJob) held_g = atomicAdd(S.gq_head, 1u);
                    if (!m_done && held_m >= (unsigned int)n_maps) { m_done = true; held_m = kNoJob; }
                    if (!g_done && held_g >= n_gjobs) { g_done = true; held_g = kNoJob; }
                    if (held_m != kNoJob) {
                        unsigned int v;
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(S.ready + held_m) : "memory");
                        if (v >= 4u) { held_m = kNoJob; continue; }  // matched where its second diagram was finished
                        if (v == 3u) { kind = 1; arg = (int)held_m; held_m = kNoJob; break; }
                    }
                    if (held_g != kNoJob) {
                        unsigned int e;
                        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(e) : "l"(S.gq + held_g / (unsigned int)Cc) : "memory");
                        if (e & kGqValid) {
                            const unsigned int ch = held_g % (unsigned int)Cc;
                            held_g = kNoJob;
                            if (e & kGqSkip) continue;  // left to grad_kernel
                            kind = 2; arg = (int)((e & kGqImage) * (unsigned int)Cc + ch);
                            break;
                        }
                    }
                    if (m_done && g_done) break;  // nothing in hand, nothing left to claim
                    __nanosleep(100);
                }
                s_kind = kind; s_arg = arg;
                if (kind == 2) s_coef = image_coef(S.cost, arg / Cc, Cc, S.ga.q, S.ga.lamda, S.ga.B_global, nullptr);
                // claim ahead: the value is not looked at before the next scheduling round
                if (kind == 1 && !m_done) held_m = atomicAdd(S.mf.counter, 1u);
                if (kind == 2 && !g_done) held_g = atomicAdd(S.gq_head, 1u);
            }
            __syncthreads();
            const int kind = s_kind, k = s_arg;
            if (kind == 0) break;
            unsigned long long tj = 0ull;
            if (S.prof && tid == 0) tj = now_ns();
            if (kind == 1) {
                // this launch's dynamic shared memory is match_one_map's kColCache-point column cache
                static_assert(kSmallSmemBytes >= kColCache * sizeof(float2), "the column cache must fit the tail's shared memory");
                const bool heavy = match_one_map(S.mf, k, reinterpret_cast<float2*>(smem));
                if (S.fuse_grad && tid == 0) map_matched(k, heavy);  // thread 0 wrote the map's cost and matched points itself
            } else {
                bar_phase = grad_job(S.ga, k, s_coef, smem, bars_s, bar_phase, S.prof ? s_gdbg : nullptr);
            }
            if (S.prof && tid == 0) {
                const unsigned long long dt = now_ns() - tj;
                if (kind == 1) { tp_match += dt; ++tp_nm; } else { tp_grad += dt; ++tp_ng; }
            }
        }
        if (tid == 0) bulk_wait_all();  // the gradient tiles this thread sent out with bulk copies are in memory
    }
    if (S.prof && tid == 0) {
        unsigned long long* o = reinterpret_cast<unsigned long long*>(S.rootpix + (size_t)blockIdx.x * S.k_stride);
        o[0] = tp_t0; o[1] = now_ns(); o[2] = tp_match; o[3] = tp_grad; o[4] = tp_nm; o[5] = tp_ng;
        if (S.fuse_match) { o[6] = s_gdbg[0]; o[7] = s_gdbg[1]; o[8] = s_gdbg[2]; o[9] = s_gdbg[3]; o[10] = s_gdbg[4]; } else o[6] = o[7] = o[8] = o[9] = o[10] = 0ull;
    }
#undef TL_PROF
}

}  // namespace tl
