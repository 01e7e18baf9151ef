// C ABI of libtopoloss.so (see include/topoloss.h for the contract and the reference
// interface each entry point replaces).  Host side: argument checks, workspace carving and
// kernel launches on the caller's stream.  No device allocation, no host synchronisation.
#include "../../include/topoloss.h"

#include <cuda_runtime.h>
#include <atomic>
#include <mutex>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "betti_kernel.cuh"
#include "diagram_kernel.cuh"
#include "dice_ce_kernel.cuh"
#include "edt_kernel.cuh"
#include "mask_kernel.cuh"
#include "match_kernel.cuh"
#include "ph_kernel.cuh"
#include "ph_small.cuh"
#include "prior_kernel.cuh"
#include "resample_kernel.cuh"
#include "seg_sort.cuh"
#include "surface_kernel.cuh"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define TL_CUDA(expr)                                                                         \
    do {                                                                                      \
        cudaError_t e_ = (expr);                                                              \
        if (e_ != cudaSuccess) return fail(TL_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_)); \
    } while (0)

constexpr int kListModeDefault = 0;  // TL_OPT_LIST_MODE when the environment does not say
// Process-wide options (tl_set_option); initial values come from the environment ONCE, at load time.
struct Options {
    std::atomic<int> v[TL_OPT_COUNT_];
    Options() {
        auto env1 = [](const char* k) { const char* e = getenv(k); return e && e[0] == '1' ? 1 : 0; };
        v[TL_OPT_FORCE_GLOBAL_KERNEL] = env1("TL_FORCE_GLOBAL");
        v[TL_OPT_PROFILE] = env1("TL_PROFILE");
        v[TL_OPT_NO_BINARY_PATH] = env1("TL_NO_BINARY");
        v[TL_OPT_WORST_CASE_WORKSPACE] = env1("TL_WORST_CASE_WORKSPACE");
        v[TL_OPT_NO_FUSED_MATCH] = env1("TL_NO_FUSED_MATCH");
        v[TL_OPT_NO_FUSED_GRAD] = env1("TL_NO_FUSED_GRAD");
        const char* lm = getenv("TL_LIST_MODE");
        v[TL_OPT_LIST_MODE] = lm ? atoi(lm) : kListModeDefault;
    }
};
Options g_opt;
inline int opt(int which) { return g_opt.v[which].load(std::memory_order_relaxed); }

// Optional per-kernel timing (bench.py's roofline): while enabled, tl_forward and tl_backward bracket each
// kernel with cudaEventRecord on the caller's stream.  Process-wide (tl_backward runs on autograd's worker
// thread), guarded by a mutex; events are created lazily and reused; nothing is synchronised until
// tl_timing_read.
constexpr int kStages = 6;        // ph, (sort: unused in the loss path), match, loss, grad fill + scatter (fused), -
constexpr int kTimingRing = 128;  // calls remembered between two reads
struct Timing {
    std::mutex mu;
    bool on = false;
    int n_fwd = 0, n_bwd = 0;
    cudaEvent_t ev[kTimingRing][kStages + 2] = {};
    bool have[kTimingRing] = {};
};
Timing g_timing;

// returns the ring slot of this call (or -1 when timing is off / the ring is full); marks are recorded under the lock
struct TimingScope {
    int call = -1;
    explicit TimingScope(bool fwd) {
        std::lock_guard<std::mutex> lk(g_timing.mu);
        if (!g_timing.on) return;
        int& n = fwd ? g_timing.n_fwd : g_timing.n_bwd;
        if (n < kTimingRing) {
            call = n;
            if (!g_timing.have[call]) {
                for (int i = 0; i < kStages + 2; ++i) cudaEventCreate(&g_timing.ev[call][i]);
                g_timing.have[call] = true;
            }
        }
        ++n;
    }
    void mark(int idx, cudaStream_t st) const { if (call >= 0) cudaEventRecord(g_timing.ev[call][idx], st); }
};

constexpr int kPhSlots = 296;      // CTAs of the global-memory persistence kernel
constexpr int kSmallSlotsMax = 160;  // per-CTA scratch slots of ph_small_kernel: one 1024-thread CTA per SM
constexpr int kSortSlots = 64;
constexpr int kMatchSlots = 296;   // tl_wasserstein
constexpr int kHeavySlotsMin = 16;  // maps whose two diagrams both exceed kSmallR points (rare with segmentation ground truth);
constexpr size_t kHeavyBytes = 32u << 20;  // scratch budget: small maps get up to kMatchSlots slots, 256 x 256 maps ~19

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

int max_pairs(int H, int W, int dim) {
    // one pair per level-0 root at most; roots are strict local extrema or mutual picks (<= nodes/2 + 1)
    const long long nn = dim == 1 ? (long long)H * W + 1 : (long long)(H + 1) * (W + 1);
    return (int)(nn / 2 + 2);
}

int sm_count() {  // per call: the device may differ between calls (one process, several GPUs)
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    return v > kSmallSlotsMax ? kSmallSlotsMax : v;
}

// STATE (kept from tl_forward to tl_backward): header, per-map bookkeeping, the pair arena.
//   header: [0] job counter (u32) | [8] arena head (u64) | [16] status (u32) | [20] heavy count (u32) |
//           [24] match work counter (u32) | [28] images published (u32) | [32] gradient jobs claimed (u32) |
//           [64..127] phase cycle counters (8 x u64)
struct StateLayout {
    int M;
    size_t counts[2], offs[2], dsum[2], cost, tpers, coef, heavy, ready, img_cnt, gq, gfused, sync_end, arena, fixed;
    unsigned long long arena_default;  // records tl_workspace_bytes asks for
};
StateLayout make_state(int M, int H, int W, int dim, int B) {
    StateLayout L;
    memset(&L, 0, sizeof(L));
    L.M = M;
    size_t o = 256;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes); return at; };
    for (int s = 0; s < 2; ++s) L.counts[s] = take(sizeof(int32_t) * (size_t)M);
    for (int s = 0; s < 2; ++s) L.offs[s] = take(sizeof(uint32_t) * (size_t)M);
    for (int s = 0; s < 2; ++s) L.dsum[s] = take(sizeof(double) * (size_t)M);
    L.cost = take(sizeof(double) * (size_t)M);
    L.tpers = take(sizeof(double) * (size_t)M);
    L.coef = take(sizeof(double) * (size_t)(B > 0 ? B : 1));
    L.heavy = take(sizeof(int32_t) * (size_t)M);
    // ready .. gfused: the launch's synchronisation words, zeroed by ONE memset per call
    L.ready = take(sizeof(uint32_t) * (size_t)M);
    L.img_cnt = take(sizeof(uint32_t) * (size_t)(B > 0 ? B : 1));
    L.gq = take(sizeof(uint32_t) * (size_t)(B > 0 ? B : 1));
    L.gfused = take(sizeof(uint32_t) * (size_t)(B > 0 ? B : 1));
    L.sync_end = o;
    L.arena = o;
    L.fixed = o;
    // Records for both sets together.  Worst case: max_pairs per map and set.  Typical: noise-like
    // predictions give ~N/5 pairs per map (iid uniform noise: N/5.1), ground truth a handful.
    const unsigned long long cap = (unsigned long long)max_pairs(H, W, dim);
    // Small maps always get (close to) the worst case: memory only matters for the big ones.
    unsigned long long typical = (unsigned long long)H * W / 5 + 64;
    if (typical < 8192) typical = 8192;
    L.arena_default = (unsigned long long)M * (opt(TL_OPT_WORST_CASE_WORKSPACE) ? 2 * cap : (typical < 2 * cap ? typical : 2 * cap));
    return L;
}

// SCRATCH (only live inside one call): per-CTA tables of the persistence kernels, the heavy matching
// path, and -- for tl_persistence_pairs -- the sort keys and the sort's buffers.
struct ScratchLayout {
    int cap, n_nodes, small, slots;
    size_t rootpix, zval, T2g, k_stride, elist, e_stride;
    size_t T, t_stride;
    size_t skeys, key_tmp, idx_a, idx_b, rec_tmp;
    size_t v, minv, u, way, pcol, used, stride_c, stride_r;
    int heavy_slots;
    size_t total;
};
ScratchLayout make_scratch(int H, int W, int dim, bool with_sort, unsigned long long arena_records) {
    ScratchLayout L;
    memset(&L, 0, sizeof(L));
    L.cap = max_pairs(H, W, dim);
    L.n_nodes = dim == 1 ? H * W + 1 : (H + 1) * (W + 1);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes); return at; };
    // shared-memory kernel: processes the map in bands of whole node columns (<= 65535 nodes each)
    // (rows are counted too: a band is at least 4 columns of ALL node rows, so n_rows <= 65535 / 4; rectangular maps)
    L.small = (W + 1) <= tl::kSmallMaxRow && (H + 1) <= tl::kSmallMaxRow && (long long)L.n_nodes < (1ll << 22);
    const bool force_global = opt(TL_OPT_FORCE_GLOBAL_KERNEL) != 0;
    if (L.small) {
        L.slots = sm_count();
        // basins per map: at most cap.  Maps of more than one band (> 65536 nodes) get tables for N/4 basins
        // unless the worst-case workspace is asked for (iid noise has N/5); overflow -> status bit + NaN loss
        size_t k_cap = (size_t)L.cap;
        // (tl_persistence_pairs, the parity-test boundary, always takes the worst case)
        if (L.n_nodes > 65537 && !opt(TL_OPT_WORST_CASE_WORKSPACE) && !with_sort) k_cap = (size_t)L.n_nodes / 4 + 2;
        L.k_stride = align_up(k_cap + 2, 64);
        L.rootpix = take(sizeof(uint32_t) * L.k_stride * L.slots);
        L.zval = take(sizeof(uint32_t) * L.k_stride * L.slots);
        L.T2g = take(sizeof(tl::TEntry) * L.k_stride * L.slots);
        // crossing edges: every node that is not a basin root owns one level-0 (non-crossing) edge, so a map
        // has at most n_edges - (n_nodes - K) of them
        const size_t n_edges = (size_t)H * (W + 1) + (size_t)(H + 1) * W;
        const size_t n_real = dim == 1 ? (size_t)H * W : (size_t)(H + 1) * (W + 1);
        L.e_stride = align_up(n_edges - n_real + L.k_stride + 64, 64);
        if (L.e_stride > align_up(n_edges, 64)) L.e_stride = align_up(n_edges, 64);
        // maps of several bands keep one band's own list at the front and the cross-band list at the back of
        // the same buffer: one band of slack (a band has < 2 * 65536 edges) keeps them apart
        if (L.n_nodes > 65537) L.e_stride += 2 * 65536 + 64;
        L.elist = take(sizeof(tl::CrossEdge) * L.e_stride * L.slots);
    }
    if (!L.small || force_global) {
        L.t_stride = align_up(sizeof(uint64_t) * (size_t)L.n_nodes) / sizeof(uint64_t);
        L.T = take(sizeof(uint64_t) * L.t_stride * kPhSlots);
    }
    if (with_sort) {
        L.skeys = take(sizeof(uint64_t) * (size_t)arena_records);
        L.key_tmp = take(sizeof(uint64_t) * (size_t)L.cap * kSortSlots);
        L.idx_a = take(sizeof(uint32_t) * (size_t)L.cap * kSortSlots);
        L.idx_b = take(sizeof(uint32_t) * (size_t)L.cap * kSortSlots);
        L.rec_tmp = take(sizeof(tl::PairRec) * (size_t)L.cap * kSortSlots);
    } else {
        L.stride_c = align_up((size_t)2 * L.cap + 2, 32);
        L.stride_r = align_up((size_t)L.cap + 2, 32);
        size_t hs = kHeavyBytes / (29 * L.stride_c);  // 8 + 8 + 4 + 4 + 1 bytes per column, 8 per row (<= half the columns)
        L.heavy_slots = (int)(hs < (size_t)kHeavySlotsMin ? (size_t)kHeavySlotsMin : hs > (size_t)kMatchSlots ? (size_t)kMatchSlots : hs);
        L.v = take(sizeof(double) * L.stride_c * L.heavy_slots);
        L.minv = take(sizeof(double) * L.stride_c * L.heavy_slots);
        L.u = take(sizeof(double) * L.stride_r * L.heavy_slots);
        L.way = take(sizeof(int32_t) * L.stride_c * L.heavy_slots);
        L.pcol = take(sizeof(int32_t) * L.stride_c * L.heavy_slots);
        L.used = take(L.stride_c * L.heavy_slots);
    }
    L.total = o > 0 ? o : 256;
    return L;
}

int check_shape(int B, int C, int H, int W, int feat_d) {
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return fail(TL_ERR_ARG, "bad shape [%d,%d,%d,%d]", B, C, H, W);
    if (feat_d != 0 && feat_d != 1) return fail(TL_ERR_ARG, "feat_d must be 0 or 1 on 2-D maps, got %d", feat_d);
    if ((long long)(2 * H + 1) * (2 * W + 1) >= 0x7FFFFFF0LL) return fail(TL_ERR_ARG, "map too large");
    if ((long long)B * C > (1 << 24)) return fail(TL_ERR_ARG, "too many maps");
    return TL_OK;
}

template <typename T>
T* at(void* ws, size_t off) { return reinterpret_cast<T*>(static_cast<char*>(ws) + off); }

tl::PairStore pair_store(void* state, const StateLayout& L, size_t state_bytes, uint64_t* skeys, float q) {
    tl::PairStore ps;
    ps.arena = at<tl::PairRec>(state, L.arena);
    ps.skeys = skeys;
    ps.head = at<unsigned long long>(state, 8);
    ps.cap = (state_bytes - L.arena) / sizeof(tl::PairRec);
    if (ps.cap > 1) --ps.cap;  // one spare record: the gradient's bulk copies read whole pairs of records
    if (ps.cap > 0xFFFFFFFFull) ps.cap = 0xFFFFFFFFull;  // offsets are 32-bit
    for (int s = 0; s < 2; ++s) {
        ps.offs[s] = at<uint32_t>(state, L.offs[s]);
        ps.counts[s] = at<int32_t>(state, L.counts[s]);
        ps.dsum[s] = at<double>(state, L.dsum[s]);
    }
    ps.status = at<unsigned int>(state, 16);
    ps.q = q;
    return ps;
}

// mf != null: the shared-memory kernel also runs the matching (tl::match_one_map) in the tail of its launch;
// *fused tells the caller whether it did (the global-memory kernel does not)
int launch_ph(const float* m0, const float* m1, int n_sets, int M, const tl::PairStore& ps, const ScratchLayout& L, int H, int W,
              int dim, void* state, void* scratch, cudaStream_t st, const tl::MatchFwdArgs* mf = nullptr, unsigned int* ready = nullptr,
              bool* fused = nullptr, const tl::GradArgs* ga = nullptr, const StateLayout* SL = nullptr) {
    if (fused) *fused = false;
    tl::PhArgs a;
    a.maps[0] = m0; a.maps[1] = m1;
    a.ps = ps;
    a.n_sets = n_sets; a.n_maps = M; a.H = H; a.W = W; a.cap = L.cap;
    a.magic_W = tl::FastDiv::magic_of((uint32_t)W); a.magic_GW = tl::FastDiv::magic_of((uint32_t)(2 * W + 1));
    a.magic_VW = tl::FastDiv::magic_of((uint32_t)(W + 1));
    a.T = at<uint64_t>(scratch, L.T); a.t_stride = L.t_stride;
    a.job_counter = at<unsigned int>(state, 0);
    TL_CUDA(cudaMemsetAsync(state, 0, 256, st));  // counters, arena head, status, phase counters
    long long jobs = (long long)n_sets * M;
    // TL_OPT_FORCE_GLOBAL_KERNEL (tests) routes every shape through the global-memory kernel, which otherwise
    // only serves maps wider than kSmallMaxRow
    const bool use_small = L.small && !opt(TL_OPT_FORCE_GLOBAL_KERNEL);
    if (use_small) {
        int grid = (int)(jobs < L.slots ? jobs : L.slots);  // one 1024-thread CTA per SM, work handed out dynamically
        tl::PhSmallArgs sa;
        sa.base = a;
        sa.rootpix = at<uint32_t>(scratch, L.rootpix); sa.zval = at<uint32_t>(scratch, L.zval);
        sa.T2g = at<tl::TEntry>(scratch, L.T2g);
        sa.k_stride = L.k_stride;
        sa.elist = at<tl::CrossEdge>(scratch, L.elist); sa.e_stride = L.e_stride;
        sa.prof = opt(TL_OPT_PROFILE) ? at<unsigned long long>(state, 64) : nullptr;
        sa.binary_path = !opt(TL_OPT_NO_BINARY_PATH);
        sa.list_mode = opt(TL_OPT_LIST_MODE);
        sa.fuse_match = mf != nullptr && !opt(TL_OPT_NO_FUSED_MATCH);
        sa.ready = ready;
        sa.fuse_grad = 0;
        memset(&sa.ga, 0, sizeof(sa.ga));
        sa.cost = nullptr; sa.img_cnt = sa.gq = sa.gq_tail = sa.gq_head = nullptr; sa.gfused = nullptr;
        if (sa.fuse_match) {
            sa.mf = *mf;
            if (SL) TL_CUDA(cudaMemsetAsync(at<char>(state, SL->ready), 0, SL->sync_end - SL->ready, st));
            else TL_CUDA(cudaMemsetAsync(ready, 0, sizeof(uint32_t) * (size_t)M, st));
            if (fused) *fused = true;
            // the gradient rides in the same tail (tl_forward_backward); the per-image counter has 16 bits per field
            if (ga && SL && ga->C <= 0xFFFF && M / ga->C <= 0xFFFFFF && !opt(TL_OPT_NO_FUSED_GRAD)) {
                sa.fuse_grad = 1;
                sa.ga = *ga;
                sa.cost = mf->cost;
                sa.img_cnt = at<unsigned int>(state, SL->img_cnt); sa.gq = at<unsigned int>(state, SL->gq);
                sa.gq_tail = at<unsigned int>(state, 28); sa.gq_head = at<unsigned int>(state, 32);
                sa.gfused = at<uint32_t>(state, SL->gfused);
            }
        } else {
            memset(&sa.mf, 0, sizeof(sa.mf));
            if (SL) TL_CUDA(cudaMemsetAsync(at<char>(state, SL->gfused), 0, SL->sync_end - SL->gfused, st));
        }
        // single band: at most 65536 pixels (H1; the last pixel doubles as OUTSIDE) / 65535 vertices (H0)
        const bool single = dim == 1 ? (long long)H * W <= 65536 : (long long)(H + 1) * (W + 1) <= 65535;
        auto launch = [&](auto kernel) -> int {
            TL_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tl::kSmallSmemBytes));
            kernel<<<grid, tl::kPhThreads, tl::kSmallSmemBytes, st>>>(sa);
            return TL_OK;
        };
        int rc;
        if (dim == 1) rc = single ? launch(tl::ph_small_kernel<1, false>) : launch(tl::ph_small_kernel<1, true>);
        else rc = single ? launch(tl::ph_small_kernel<0, false>) : launch(tl::ph_small_kernel<0, true>);
        if (rc != TL_OK) return rc;
    } else {
        if (SL) TL_CUDA(cudaMemsetAsync(at<char>(state, SL->gfused), 0, SL->sync_end - SL->gfused, st));
        const int grid = (int)(jobs < kPhSlots ? jobs : kPhSlots);
        if (dim == 1) tl::ph_kernel<1><<<grid, tl::kPhThreads, 0, st>>>(a);
        else tl::ph_kernel<0><<<grid, tl::kPhThreads, 0, st>>>(a);
    }
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

void fill_match_scratch(tl::MatchArgs& a, void* ws, size_t v, size_t minv, size_t u, size_t way, size_t pcol,
                        size_t used, size_t stride_c, size_t stride_r) {
    a.v = at<double>(ws, v); a.minv = at<double>(ws, minv); a.u = at<double>(ws, u);
    a.way = at<int32_t>(ws, way); a.pcol = at<int32_t>(ws, pcol); a.used = at<uint8_t>(ws, used);
    a.stride_c = stride_c; a.stride_r = stride_r;
}

}  // namespace

extern "C" {

int tl_version(void) { return TL_ABI_VERSION; }

const char* tl_last_error(void) { return g_err; }

int tl_set_option(int which, int value) {
    if (which < 0 || which >= TL_OPT_COUNT_) return fail(TL_ERR_ARG, "unknown option %d", which);
    g_opt.v[which].store(value, std::memory_order_relaxed);
    return TL_OK;
}

int tl_get_option(int which) {
    if (which < 0 || which >= TL_OPT_COUNT_) return fail(TL_ERR_ARG, "unknown option %d", which);
    return opt(which);
}

/* Debug aid (not part of the hot path): copies the 8 phase cycle counters that the persistence
 * kernel accumulates while TL_OPT_PROFILE is set.  Synchronises the device. */
int tl_debug_profile(const void* state, unsigned long long* host_out8) {
    if (!state || !host_out8) return fail(TL_ERR_ARG, "null pointer");
    TL_CUDA(cudaDeviceSynchronize());
    TL_CUDA(cudaMemcpy(host_out8, static_cast<const char*>(state) + 64, 64, cudaMemcpyDeviceToHost));
    return TL_OK;
}

int tl_debug_tail_profile(const void* scratch, int H, int W, int feat_d, unsigned long long* host_out, int max_slots) {
    if (!scratch || !host_out || max_slots <= 0) return fail(TL_ERR_ARG, "null pointer");
    const ScratchLayout L = make_scratch(H, W, feat_d, false, 0);
    if (!L.small) return fail(TL_ERR_ARG, "shape not served by the shared-memory kernel");
    TL_CUDA(cudaDeviceSynchronize());
    const int n = L.slots < max_slots ? L.slots : max_slots;
    for (int i = 0; i < n; ++i)
        TL_CUDA(cudaMemcpy(host_out + 11 * i, static_cast<const char*>(scratch) + L.rootpix + sizeof(uint32_t) * L.k_stride * i, 88, cudaMemcpyDeviceToHost));
    return n;
}

int tl_status(const void* state, int* host_status, void* stream) {
    if (!state || !host_status) return fail(TL_ERR_ARG, "null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned int v = 0;
    TL_CUDA(cudaMemcpyAsync(&v, static_cast<const char*>(state) + 16, 4, cudaMemcpyDeviceToHost, st));
    TL_CUDA(cudaStreamSynchronize(st));
    *host_status = (int)v;
    return TL_OK;
}

int tl_timing_enable(int on) {
    std::lock_guard<std::mutex> lk(g_timing.mu);
    g_timing.on = on != 0;
    g_timing.n_fwd = g_timing.n_bwd = 0;
    return TL_OK;
}

int tl_timing_read(float* ms_sum6, int* n_calls) {
    if (!ms_sum6 || !n_calls) return fail(TL_ERR_ARG, "null pointer");
    std::lock_guard<std::mutex> lk(g_timing.mu);
    Timing& t = g_timing;
    for (int i = 0; i < kStages; ++i) ms_sum6[i] = 0.f;
    const int nf = t.n_fwd < kTimingRing ? t.n_fwd : kTimingRing;
    const int nb = t.n_bwd < kTimingRing ? t.n_bwd : kTimingRing;
    for (int c = 0; c < nf; ++c) {
        TL_CUDA(cudaEventSynchronize(t.ev[c][4]));
        for (int i = 0; i < 4; ++i) { float ms = 0.f; TL_CUDA(cudaEventElapsedTime(&ms, t.ev[c][i], t.ev[c][i + 1])); ms_sum6[i] += ms; }
    }
    for (int c = 0; c < nb; ++c) {
        TL_CUDA(cudaEventSynchronize(t.ev[c][7]));
        for (int i = 4; i < 6; ++i) { float ms = 0.f; TL_CUDA(cudaEventElapsedTime(&ms, t.ev[c][i + 1], t.ev[c][i + 2])); ms_sum6[i] += ms; }
    }
    n_calls[0] = nf; n_calls[1] = nb;
    t.n_fwd = t.n_bwd = 0;
    return TL_OK;
}

#ifdef TL_STATS
int tl_debug_stats(unsigned long long* host_out8, int reset) {
    TL_CUDA(cudaDeviceSynchronize());
    TL_CUDA(cudaMemcpyFromSymbol(host_out8, tl::g_stats, 64));
    if (reset) { unsigned long long z[8] = {0}; TL_CUDA(cudaMemcpyToSymbol(tl::g_stats, z, 64)); }
    return TL_OK;
}
#endif

int tl_max_pairs(int H, int W, int dim) {
    if (H <= 0 || W <= 0 || (dim != 0 && dim != 1)) return fail(TL_ERR_ARG, "bad arguments");
    return max_pairs(H, W, dim);
}

int tl_workspace_bytes(int B, int C, int H, int W, int feat_d, size_t* state_bytes, size_t* scratch_bytes) {
    if (!state_bytes || !scratch_bytes) return fail(TL_ERR_ARG, "null pointer");
    int rc = check_shape(B, C, H, W, feat_d);
    if (rc != TL_OK) return rc;
    const StateLayout S = make_state(B * C, H, W, feat_d, B);
    *state_bytes = S.fixed + (size_t)S.arena_default * sizeof(tl::PairRec);
    *scratch_bytes = make_scratch(H, W, feat_d, false, 0).total;
    return TL_OK;
}

// tl_forward (grad_pred == null) and tl_forward_backward: grad_pred, when given, receives d loss / d pred for an
// upstream gradient of 1 -- written in the tail of the persistence launch for every image the small-R matching
// served, by grad_kernel afterwards for the rest
static int forward_impl(const float* pred, const float* truth, int B, int C, int H, int W, int feat_d, float q,
                        float lamda, int loss_r, int B_global, void* state, size_t state_bytes, void* scratch,
                        size_t scratch_bytes, float* loss_out, float* grad_pred, void* stream) {
    int rc = check_shape(B, C, H, W, feat_d);
    if (rc != TL_OK) return rc;
    if (!pred || !truth || !state || !scratch || !loss_out) return fail(TL_ERR_ARG, "null pointer");
    if (!(q > 0.f)) return fail(TL_ERR_ARG, "loss_q must be positive");
    if (B_global <= 0) B_global = B;
    const int M = B * C;
    const StateLayout S = make_state(M, H, W, feat_d, B);
    const ScratchLayout L = make_scratch(H, W, feat_d, false, 0);
    if (state_bytes < S.fixed + sizeof(tl::PairRec)) return fail(TL_ERR_WORKSPACE, "state %zu < %zu bytes", state_bytes, S.fixed + sizeof(tl::PairRec));
    if (scratch_bytes < L.total) return fail(TL_ERR_WORKSPACE, "scratch %zu < %zu bytes", scratch_bytes, L.total);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const tl::PairStore ps = pair_store(state, S, state_bytes, nullptr, q);

    tl::GradArgs g;
    g.arena = at<tl::PairRec>(state, S.arena); g.offs = at<uint32_t>(state, S.offs[0]); g.counts = at<int32_t>(state, S.counts[0]);
    g.coef = at<double>(state, S.coef); g.grad_loss = nullptr;
    g.M = M; g.C = C; g.N = H * W; g.B_global = B_global; g.loss_r = loss_r;
    g.q = q; g.lamda = lamda; g.grad_pred = grad_pred; g.gfused = at<uint32_t>(state, S.gfused);

    bool fused = false;
    {
    const TimingScope tm(true);
    tm.mark(0, st);
    // pairs leave the persistence kernel in a deterministic (raster) order, so the matching needs no
    // sort; the segmented sort only serves tl_persistence_pairs (gudhi's emission order)
    tl::MatchFwdArgs mf;
    mf.ps = ps; mf.n_maps = M; mf.loss_r = loss_r; mf.q = q;
    mf.cost = at<double>(state, S.cost); mf.tpers = at<double>(state, S.tpers);
    mf.heavy = at<int32_t>(state, S.heavy); mf.n_heavy = at<unsigned int>(state, 20);
    mf.counter = at<unsigned int>(state, 24);
    rc = launch_ph(pred, truth, 2, M, ps, L, H, W, feat_d, state, scratch, st, &mf, at<unsigned int>(state, S.ready), &fused,
                   grad_pred ? &g : nullptr, &S);
    if (rc != TL_OK) return rc;
    tm.mark(1, st);
    tm.mark(2, st);
    if (!fused) {  // global-memory persistence kernel (or the fusion switched off): the matching gets its own launch
        TL_CUDA(cudaFuncSetAttribute(tl::match_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tl::kColCache * 8));
        tl::match_small_kernel<<<M < kMatchSlots ? M : kMatchSlots, tl::kMatchThreads, tl::kColCache * 8, st>>>(mf);
        TL_CUDA(cudaGetLastError());
    }
    {   // maps with two large diagrams (none for segmentation ground truth): general kernel, global scratch
        tl::MatchArgs m;
        const char* recs = reinterpret_cast<const char*>(ps.arena) + offsetof(tl::PairRec, b);
        m.d1 = tl::Diagrams{recs, (int)sizeof(tl::PairRec), nullptr, ps.offs[0], ps.counts[0]};
        m.d2 = tl::Diagrams{recs, (int)sizeof(tl::PairRec), nullptr, ps.offs[1], ps.counts[1]};
        m.n_diag = M; m.q = q; m.loss_r = 0;
        m.cost = mf.cost; m.tpers = nullptr; m.match1 = nullptr; m.fill1 = ps.arena;
        m.list = mf.heavy; m.n_list = mf.n_heavy;
        fill_match_scratch(m, scratch, L.v, L.minv, L.u, L.way, L.pcol, L.used, L.stride_c, L.stride_r);
        m.counter = nullptr;
        tl::match_kernel<<<M < L.heavy_slots ? M : L.heavy_slots, tl::kMatchThreads, 0, st>>>(m);
        TL_CUDA(cudaGetLastError());
    }
    tm.mark(3, st);

    tl::LossArgs la;
    la.cost = mf.cost; la.tpers = mf.tpers; la.B = B; la.C = C; la.B_global = B_global; la.loss_r = loss_r;
    la.q = q; la.lamda = lamda; la.loss_out = loss_out; la.coef = at<double>(state, S.coef);
    la.status = ps.status;
    tl::loss_kernel<<<1, 256, 0, st>>>(la);
    TL_CUDA(cudaGetLastError());
    tm.mark(4, st);
    }
    if (grad_pred) {  // whatever the tail did not serve (all of it when the fusion is off)
        const TimingScope tm(false);
        tm.mark(5, st);
        tm.mark(6, st);
        // (with the gradient fused into the persistence launch this only serves images with maps on the heavy list:
        // a small grid, its CTAs mostly look at gfused[] and leave)
        const bool in_tail = fused && C <= 0xFFFF && B <= 0xFFFFFF && !opt(TL_OPT_NO_FUSED_GRAD);
        const int cap = in_tail ? 296 : 1184;
        tl::grad_kernel<<<M < cap ? M : cap, 512, 0, st>>>(g);
        TL_CUDA(cudaGetLastError());
        tm.mark(7, st);
    }
    return TL_OK;
}

int tl_forward(const float* pred, const float* truth, int B, int C, int H, int W, int feat_d, float q,
               float lamda, int loss_r, int B_global, void* state, size_t state_bytes, void* scratch,
               size_t scratch_bytes, float* loss_out, void* stream) {
    return forward_impl(pred, truth, B, C, H, W, feat_d, q, lamda, loss_r, B_global, state, state_bytes, scratch,
                        scratch_bytes, loss_out, nullptr, stream);
}

int tl_forward_backward(const float* pred, const float* truth, int B, int C, int H, int W, int feat_d, float q,
                        float lamda, int loss_r, int B_global, void* state, size_t state_bytes, void* scratch,
                        size_t scratch_bytes, float* loss_out, float* grad_pred, void* stream) {
    if (!grad_pred) return fail(TL_ERR_ARG, "null pointer");
    return forward_impl(pred, truth, B, C, H, W, feat_d, q, lamda, loss_r, B_global, state, state_bytes, scratch,
                        scratch_bytes, loss_out, grad_pred, stream);
}

int tl_unpack_mask_bits(const uint8_t* bits, float* maps, long long n_pixels, void* stream) {
    if (!bits || !maps || n_pixels < 0 || (n_pixels & 7)) return fail(TL_ERR_ARG, "n_pixels must be a non-negative multiple of 8");
    if (n_pixels == 0) return TL_OK;
    const long long n_bytes = n_pixels >> 3;
    long long blocks = (n_bytes / 4 + 255) / 256;
    if (blocks > 2368) blocks = 2368;
    if (blocks < 1) blocks = 1;
    tl::unpack_bits_kernel<<<(int)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(bits, maps, n_bytes);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_scale_gradient(const float* grad_loss, float* grad_pred, long long n, void* stream) {
    if (!grad_pred || n < 0) return fail(TL_ERR_ARG, "bad argument");
    if (!grad_loss || n == 0) return TL_OK;  // NULL: upstream gradient 1.0
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    long long blocks = (n / 4 + 255) / 256;
    if (blocks > 1184) blocks = 1184;
    if (blocks < 1) blocks = 1;
    tl::scale_kernel<<<(int)blocks, 256, 0, st>>>(grad_loss, grad_pred, n);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_backward(const float* grad_loss, const void* state, size_t state_bytes, int B, int C, int H, int W,
                int feat_d, float q, float lamda, int loss_r, int B_global, float* grad_pred, void* stream) {
    int rc = check_shape(B, C, H, W, feat_d);
    if (rc != TL_OK) return rc;
    if (!state || !grad_pred) return fail(TL_ERR_ARG, "null pointer");
    if (B_global <= 0) B_global = B;
    const int M = B * C;
    const StateLayout S = make_state(M, H, W, feat_d, B);
    if (state_bytes < S.fixed + sizeof(tl::PairRec)) return fail(TL_ERR_WORKSPACE, "state %zu < %zu bytes", state_bytes, S.fixed + sizeof(tl::PairRec));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    void* w = const_cast<void*>(state);
    const TimingScope tm(false);
    tm.mark(5, st);
    tm.mark(6, st);
    tl::GradArgs g;
    g.arena = at<tl::PairRec>(w, S.arena); g.offs = at<uint32_t>(w, S.offs[0]); g.counts = at<int32_t>(w, S.counts[0]);
    g.coef = at<double>(w, S.coef); g.grad_loss = grad_loss;
    g.M = M; g.C = C; g.N = H * W; g.B_global = B_global; g.loss_r = loss_r;
    g.q = q; g.lamda = lamda; g.grad_pred = grad_pred; g.gfused = nullptr;  // always the full gradient
    tl::grad_kernel<<<M < 1184 ? M : 1184, 512, 0, st>>>(g);
    TL_CUDA(cudaGetLastError());
    tm.mark(7, st);
    return TL_OK;
}

}  // extern "C"

namespace {

__global__ void export_pairs_kernel(tl::PairStore ps, int n_maps, int32_t* pairs, int cap_out, int32_t* counts) {
    for (int map = blockIdx.x; map < n_maps; map += gridDim.x) {
        const int n = ps.counts[0][map];
        if (threadIdx.x == 0) counts[map] = n;
        const tl::PairRec* recs = ps.arena + ps.offs[0][map];
        const int lim = min(n, cap_out);
        for (int i = threadIdx.x; i < lim; i += blockDim.x) {
            const tl::PairRec r = recs[i];
            pairs[((size_t)map * cap_out + i) * 2] = r.cre;
            pairs[((size_t)map * cap_out + i) * 2 + 1] = r.des;
        }
    }
}

// tl_persistence_pairs keeps everything in ONE buffer: [state | scratch]
struct PairsLayout { StateLayout S; ScratchLayout L; size_t state_bytes, scratch_off, total; };
PairsLayout make_pairs_layout(int n_maps, int H, int W, int dim) {
    PairsLayout P;
    P.S = make_state(n_maps, H, W, dim, n_maps);
    // one set only, and the caller may look at pathological maps: worst-case record count, capped at 2^32 - 1
    unsigned long long recs = (unsigned long long)n_maps * (unsigned long long)max_pairs(H, W, dim);
    if (!opt(TL_OPT_WORST_CASE_WORKSPACE) && recs > (1ull << 28)) recs = 1ull << 28;  // 6 GiB of records
    if (recs > 0xFFFFFFFFull) recs = 0xFFFFFFFFull;
    P.state_bytes = align_up(P.S.fixed + (size_t)recs * sizeof(tl::PairRec));
    P.L = make_scratch(H, W, dim, true, recs);
    P.scratch_off = P.state_bytes;
    P.total = P.state_bytes + P.L.total;
    return P;
}

// The persistence launch for one set of maps, then the segmented sort into gudhi's emission order: the pairs of
// map i are records ps.offs[0][i] .. + ps.counts[0][i] of the arena in `state` (P.state_bytes of layout P.S);
// `scratch` holds P.L (the persistence tables, the sort keys and the sort's buffers)
int sorted_pairs(const float* maps, int n_maps, int H, int W, int dim, void* state, void* scratch, const PairsLayout& P,
                 cudaStream_t st, tl::PairStore* ps_out) {
    const tl::PairStore ps = pair_store(state, P.S, P.state_bytes, at<uint64_t>(scratch, P.L.skeys), 2.0f);
    int rc = launch_ph(maps, nullptr, 1, n_maps, ps, P.L, H, W, dim, state, scratch, st);
    if (rc != TL_OK) return rc;
    tl::SortArgs a;
    a.ps = ps; a.n_sets = 1; a.n_maps = n_maps; a.cap = P.L.cap;
    a.key_tmp = at<uint64_t>(scratch, P.L.key_tmp);
    a.idx_a = at<uint32_t>(scratch, P.L.idx_a);
    a.idx_b = at<uint32_t>(scratch, P.L.idx_b);
    a.rec_tmp = at<tl::PairRec>(scratch, P.L.rec_tmp);
    tl::seg_sort_kernel<<<n_maps < kSortSlots ? n_maps : kSortSlots, tl::kSortThreads, 0, st>>>(a);
    TL_CUDA(cudaGetLastError());
    *ps_out = ps;
    return TL_OK;
}

// [rows][2] buffers are read and written as int2 / float2: they must be 8-byte aligned (a null pointer passes)
inline bool misaligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7) != 0; }

// argument checks shared by tl_diagrams_compute / tl_diagrams_gather; the packed offsets are int32
int diagrams_args(int n_maps, int H, int W, int dim, const void* ws, size_t ws_bytes, PairsLayout* P) {
    int rc = check_shape(n_maps, 1, H, W, dim);
    if (rc != TL_OK) return rc;
    if (!ws) return fail(TL_ERR_ARG, "null pointer");
    *P = make_pairs_layout(n_maps, H, W, dim);
    if (ws_bytes < P->total) return fail(TL_ERR_ARG, "workspace %zu < %zu bytes (tl_diagrams_workspace_bytes)", ws_bytes, P->total);
    if ((P->state_bytes - P->S.fixed) / sizeof(tl::PairRec) > 0x7FFFFFFFull)
        return fail(TL_ERR_ARG, "%d maps of %dx%d can hold more pairs than int32 offsets address", n_maps, H, W);
    return TL_OK;
}

}  // namespace

extern "C" {

int tl_pairs_workspace_bytes(int n_maps, int H, int W, int dim, size_t* bytes) {
    if (!bytes) return fail(TL_ERR_ARG, "bytes is null");
    int rc = check_shape(n_maps, 1, H, W, dim);
    if (rc != TL_OK) return rc;
    *bytes = make_pairs_layout(n_maps, H, W, dim).total;
    return TL_OK;
}

int tl_persistence_pairs(const float* maps, int n_maps, int H, int W, int dim, void* ws, size_t ws_bytes,
                         int32_t* pairs, int cap, int32_t* counts, void* stream) {
    int rc = check_shape(n_maps, 1, H, W, dim);
    if (rc != TL_OK) return rc;
    if (!maps || !ws || !pairs || !counts || cap <= 0) return fail(TL_ERR_ARG, "null pointer or cap <= 0");
    const PairsLayout P = make_pairs_layout(n_maps, H, W, dim);
    if (ws_bytes < P.total) return fail(TL_ERR_WORKSPACE, "workspace %zu < %zu bytes", ws_bytes, P.total);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    tl::PairStore ps;
    rc = sorted_pairs(maps, n_maps, H, W, dim, ws, static_cast<char*>(ws) + P.scratch_off, P, st, &ps);
    if (rc != TL_OK) return rc;
    export_pairs_kernel<<<n_maps < 1184 ? n_maps : 1184, 256, 0, st>>>(ps, n_maps, pairs, cap, counts);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

// ---- persistence diagrams as packed, differentiable tensors (tl_diagrams_*)

int tl_diagrams_workspace_bytes(int n_maps, int H, int W, int dim, size_t* bytes) {
    if (!bytes) return fail(TL_ERR_ARG, "bytes is null");
    int rc = check_shape(n_maps, 1, H, W, dim);
    if (rc != TL_OK) return rc;
    *bytes = make_pairs_layout(n_maps, H, W, dim).total;
    return TL_OK;
}

int tl_diagrams_compute(const float* maps, int n_maps, int H, int W, int dim, void* ws, size_t ws_bytes,
                        int32_t* offsets, int32_t* status, void* stream) {
    PairsLayout P;
    int rc = diagrams_args(n_maps, H, W, dim, ws, ws_bytes, &P);
    if (rc != TL_OK) return rc;
    if (!maps || !offsets) return fail(TL_ERR_ARG, "null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    tl::PairStore ps;
    rc = sorted_pairs(maps, n_maps, H, W, dim, ws, static_cast<char*>(ws) + P.scratch_off, P, st, &ps);
    if (rc != TL_OK) return rc;
    tl::diagram_offsets_kernel<<<1, tl::kScanThreads, 0, st>>>(ps.counts[0], n_maps, ps.status, offsets, status);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_diagrams_gather(const float* maps, int n_maps, int H, int W, int dim, const void* ws, size_t ws_bytes,
                       const int32_t* offsets, const int32_t* host_offsets, long long P, int32_t* pairs, float* diagram,
                       void* stream) {
    PairsLayout L;
    int rc = diagrams_args(n_maps, H, W, dim, ws, ws_bytes, &L);
    if (rc != TL_OK) return rc;
    if (!maps || !offsets || !host_offsets) return fail(TL_ERR_ARG, "null pointer");
    if (P < 0 || (P > 0 && (!pairs || !diagram))) return fail(TL_ERR_ARG, "null output buffer for %lld pairs", P);
    if (misaligned8(pairs) || misaligned8(diagram)) return fail(TL_ERR_ARG, "pairs and diagram must be 8-byte aligned");
    if (host_offsets[0] != 0) return fail(TL_ERR_ARG, "offsets[0] = %d, not 0", host_offsets[0]);
    for (int i = 0; i < n_maps; ++i)
        if (host_offsets[i + 1] < host_offsets[i]) return fail(TL_ERR_ARG, "offsets decrease at map %d", i);
    if ((long long)host_offsets[n_maps] != P) return fail(TL_ERR_ARG, "P = %lld disagrees with offsets[%d] = %d", P, n_maps, host_offsets[n_maps]);
    if (P == 0) return TL_OK;
    void* w = const_cast<void*>(ws);
    const int grid = n_maps < 1184 ? n_maps : 1184;
    tl::diagram_gather_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        at<tl::PairRec>(w, L.S.arena), at<uint32_t>(w, L.S.offs[0]), maps, (long long)H * W, n_maps, offsets,
        reinterpret_cast<int2*>(pairs), reinterpret_cast<float2*>(diagram));
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_diagrams_backward(const int32_t* pairs, const int32_t* offsets, const float* grad_diagram, long long P,
                         int n_maps, int H, int W, float* grad_maps, void* stream) {
    if (n_maps <= 0 || H <= 0 || W <= 0 || (long long)H * W >= 0x7FFFFFF0LL) return fail(TL_ERR_ARG, "bad shape [%d,%d,%d]", n_maps, H, W);
    if (P < 0 || !offsets || !grad_maps || (P > 0 && (!pairs || !grad_diagram))) return fail(TL_ERR_ARG, "null pointer");
    if (misaligned8(pairs) || misaligned8(grad_diagram)) return fail(TL_ERR_ARG, "pairs and grad_diagram must be 8-byte aligned");
    const int grid = n_maps < 1184 ? n_maps : 1184;
    tl::diagram_backward_kernel<<<grid, 512, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const int2*>(pairs), offsets, reinterpret_cast<const float2*>(grad_diagram), n_maps, H * W, grad_maps);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_wasserstein_backward(const float* D1, const int32_t* off1, const float* D2, const int32_t* off2, int n_diag,
                            float q, const int32_t* match1, const float* grad_cost, float* grad_D1, float* grad_D2,
                            void* stream) {
    if (n_diag <= 0) return fail(TL_ERR_ARG, "n_diag must be positive, got %d", n_diag);
    if (!D1 || !off1 || !D2 || !off2 || !match1 || !grad_cost) return fail(TL_ERR_ARG, "null pointer");
    if (!(q > 0.f)) return fail(TL_ERR_ARG, "q must be positive");
    if (misaligned8(D1) || misaligned8(D2) || misaligned8(grad_D1) || misaligned8(grad_D2))
        return fail(TL_ERR_ARG, "D1, D2, grad_D1 and grad_D2 must be 8-byte aligned");
    if (!grad_D1 && !grad_D2) return TL_OK;
    tl::WassersteinBwdArgs a;
    a.d1 = reinterpret_cast<const float2*>(D1); a.off1 = off1;
    a.d2 = reinterpret_cast<const float2*>(D2); a.off2 = off2;
    a.n_diag = n_diag; a.q = q; a.match1 = match1; a.grad_cost = grad_cost;
    a.g1 = reinterpret_cast<float2*>(grad_D1); a.g2 = reinterpret_cast<float2*>(grad_D2);
    tl::wasserstein_backward_kernel<<<n_diag < 1184 ? n_diag : 1184, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_wasserstein_workspace_bytes(int n_diag, int max_rows1, int max_rows2, size_t* bytes) {
    if (!bytes || n_diag <= 0 || max_rows1 < 0 || max_rows2 < 0) return fail(TL_ERR_ARG, "bad arguments");
    const size_t sc = align_up((size_t)max_rows1 + max_rows2 + 2, 32);
    const size_t sr = align_up((size_t)(max_rows1 < max_rows2 ? max_rows1 : max_rows2) + 2, 32);
    const int slots = n_diag < kMatchSlots ? n_diag : kMatchSlots;
    *bytes = align_up(sizeof(double) * sc * slots) * 2 + align_up(sizeof(double) * sr * slots) +
             align_up(sizeof(int32_t) * sc * slots) * 2 + align_up(sc * slots);
    return TL_OK;
}

int tl_wasserstein(const float* D1, const int32_t* off1, const float* D2, const int32_t* off2, int n_diag,
                   int max_rows1, int max_rows2, float q, void* ws, size_t ws_bytes, double* cost,
                   int32_t* match1, void* stream) {
    size_t need = 0;
    int rc = tl_wasserstein_workspace_bytes(n_diag, max_rows1, max_rows2, &need);
    if (rc != TL_OK) return rc;
    if (!D1 || !off1 || !D2 || !off2 || !ws || !cost || !match1) return fail(TL_ERR_ARG, "null pointer");
    if (!(q > 0.f)) return fail(TL_ERR_ARG, "q must be positive");
    if (ws_bytes < need) return fail(TL_ERR_WORKSPACE, "workspace %zu < %zu bytes", ws_bytes, need);
    const size_t sc = align_up((size_t)max_rows1 + max_rows2 + 2, 32);
    const size_t sr = align_up((size_t)(max_rows1 < max_rows2 ? max_rows1 : max_rows2) + 2, 32);
    const int slots = n_diag < kMatchSlots ? n_diag : kMatchSlots;
    size_t o = 0;
    auto take = [&](size_t b) { size_t a = o; o += align_up(b); return a; };
    const size_t ov = take(sizeof(double) * sc * slots), ominv = take(sizeof(double) * sc * slots);
    const size_t ou = take(sizeof(double) * sr * slots);
    const size_t oway = take(sizeof(int32_t) * sc * slots), opcol = take(sizeof(int32_t) * sc * slots);
    const size_t oused = take(sc * slots);
    tl::MatchArgs m;
    m.d1 = tl::Diagrams{reinterpret_cast<const char*>(D1), 8, off1, nullptr, nullptr};
    m.d2 = tl::Diagrams{reinterpret_cast<const char*>(D2), 8, off2, nullptr, nullptr};
    m.n_diag = n_diag; m.q = q; m.loss_r = 0; m.cost = cost; m.tpers = nullptr; m.match1 = match1; m.fill1 = nullptr;
    m.counter = nullptr; m.list = nullptr; m.n_list = nullptr;
    fill_match_scratch(m, ws, ov, ominv, ou, oway, opcol, oused, sc, sr);
    tl::match_kernel<<<slots, tl::kMatchThreads, 0, static_cast<cudaStream_t>(stream)>>>(m);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

}  // extern "C"

extern "C" {

namespace {
int resample_args(tl::ResampleArgs& a, const float* in, int n_maps, int H, int W, int S, int apply_sigmoid) {
    if (!in) return fail(TL_ERR_ARG, "null pointer");
    if (n_maps <= 0 || H <= 0 || W <= 0 || S <= 0) return fail(TL_ERR_ARG, "bad shape [%d,%d,%d] -> %d", n_maps, H, W, S);
    if ((long long)n_maps * H * W >= (1ll << 40) || (long long)n_maps * S * S >= (1ll << 40)) return fail(TL_ERR_ARG, "too large");
    a.in = in; a.out = nullptr; a.gout = nullptr; a.gin = nullptr;
    a.n_maps = n_maps; a.H = H; a.W = W; a.S = S; a.apply_sigmoid = apply_sigmoid != 0;
    a.sy = S > 1 ? (float)(H - 1) / (float)(S - 1) : 0.f;
    a.sx = S > 1 ? (float)(W - 1) / (float)(S - 1) : 0.f;
    return TL_OK;
}
int grid_for(long long work, int block) {
    long long g = (work + block - 1) / block;
    const long long cap = 148ll * 16;  // a few waves of resident CTAs on a 148-SM B200, grid-stride beyond
    return (int)(g < 1 ? 1 : g > cap ? cap : g);
}
}  // namespace

int tl_resample_forward(const float* in, int n_maps, int H, int W, int S, int apply_sigmoid, float* out, void* stream) {
    tl::ResampleArgs a;
    int rc = resample_args(a, in, n_maps, H, W, S, apply_sigmoid);
    if (rc != TL_OK) return rc;
    if (!out) return fail(TL_ERR_ARG, "null pointer");
    a.out = out;
    tl::resample_fwd_kernel<<<grid_for((long long)n_maps * S * S, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_resample_backward(const float* grad_out, const float* in, int n_maps, int H, int W, int S, int apply_sigmoid,
                         float* grad_in, void* stream) {
    tl::ResampleArgs a;
    int rc = resample_args(a, in, n_maps, H, W, S, apply_sigmoid);
    if (rc != TL_OK) return rc;
    if (!grad_out || !grad_in) return fail(TL_ERR_ARG, "null pointer");
    if (reinterpret_cast<uintptr_t>(grad_in) & 15) return fail(TL_ERR_ARG, "grad_in must be 16-byte aligned");
    a.gout = grad_out; a.gin = grad_in;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long n = (long long)n_maps * H * W;
    tl::zero_fill_kernel<<<grid_for(n >> 2, 256), 256, 0, st>>>(grad_in, n);
    TL_CUDA(cudaGetLastError());
    tl::resample_bwd_kernel<<<grid_for((long long)n_maps * S * S, 256), 256, 0, st>>>(a);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

}  // extern "C"

extern "C" {

namespace {
int post_args(tl::PostArgs& a, int n_maps, int Hs, int Ws, int T, int rh, int rw, int oh, int ow) {
    if (n_maps <= 0 || Hs <= 0 || Ws <= 0 || T <= 0 || oh <= 0 || ow <= 0) return fail(TL_ERR_ARG, "bad shape");
    if (rh <= 0 || rw <= 0 || rh > T || rw > T) return fail(TL_ERR_ARG, "crop [%d,%d] outside the %dx%d intermediate", rh, rw, T, T);
    if ((long long)n_maps * oh * ow >= (1ll << 40)) return fail(TL_ERR_ARG, "too large");
    a.in = nullptr; a.out = nullptr; a.gout = nullptr; a.gin = nullptr;
    a.n_maps = n_maps; a.Hs = Hs; a.Ws = Ws; a.T = T; a.rh = rh; a.rw = rw; a.oh = oh; a.ow = ow;
    a.s1y = (float)Hs / (float)T; a.s1x = (float)Ws / (float)T;
    a.s2y = (float)rh / (float)oh; a.s2x = (float)rw / (float)ow;
    return TL_OK;
}
}  // namespace

int tl_postprocess_forward(const float* in, int n_maps, int Hs, int Ws, int T, int rh, int rw, int oh, int ow,
                           float* out, void* stream) {
    tl::PostArgs a;
    int rc = post_args(a, n_maps, Hs, Ws, T, rh, rw, oh, ow);
    if (rc != TL_OK) return rc;
    if (!in || !out) return fail(TL_ERR_ARG, "null pointer");
    a.in = in; a.out = out;
    const int ftx = (ow + tl::kFwdCols - 1) / tl::kFwdCols, fty = (oh + tl::kFwdRows - 1) / tl::kFwdRows;
    const long long f_tiles = (long long)n_maps * fty * ftx, f_cap = 148ll * 64;
    tl::postprocess_fwd_kernel<<<(int)(f_tiles < f_cap ? f_tiles : f_cap), tl::kFwdCols, 0, static_cast<cudaStream_t>(stream)>>>(a, fty, ftx);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_postprocess_backward(const float* grad_out, int n_maps, int Hs, int Ws, int T, int rh, int rw, int oh, int ow,
                            float* grad_in, void* stream) {
    tl::PostArgs a;
    int rc = post_args(a, n_maps, Hs, Ws, T, rh, rw, oh, ow);
    if (rc != TL_OK) return rc;
    if (!grad_out || !grad_in) return fail(TL_ERR_ARG, "null pointer");
    if (reinterpret_cast<uintptr_t>(grad_in) & 15) return fail(TL_ERR_ARG, "grad_in must be 16-byte aligned");
    a.gout = grad_out; a.gin = grad_in;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    // taps per source pixel and axis: 2 * (out / mid) * (T / src) + 3.  Few (the reference down-samples to the
    // original size): gather kernel, every source pixel written once.  Many (strong up-sampling): scatter kernel.
    const double ky = 2.0 * oh * T / ((double)Hs * rh) + 3.0, kx = 2.0 * ow * T / ((double)Ws * rw) + 3.0;
    if (ky <= tl::kGK && kx <= tl::kGK) {
        const int gcy = (Hs + tl::kGRows - 1) / tl::kGRows, gtx = (Ws + tl::kGT_X - 1) / tl::kGT_X;
        // a CTA keeps one strip position (gcy * gtx of them) and walks over maps: grid = positions x map lanes
        const int classes = gcy * gtx;
        int lanes = (148 * 10 + classes - 1) / classes;
        if (lanes > n_maps) lanes = n_maps;
        if (lanes < 1) lanes = 1;
        tl::postprocess_bwd_gather_kernel<<<classes * lanes, tl::kGT_Y * tl::kGT_X, 0, st>>>(a, gcy, gtx);
        TL_CUDA(cudaGetLastError());
        return TL_OK;
    }
    const long long n = (long long)n_maps * Hs * Ws;
    tl::zero_fill_kernel<<<grid_for(n >> 2, 256), 256, 0, st>>>(grad_in, n);
    TL_CUDA(cudaGetLastError());
    const int tiles_y = (oh + tl::kPostTileY - 1) / tl::kPostTileY, tiles_x = (ow + tl::kPostTileX - 1) / tl::kPostTileX;
    const long long n_tiles = (long long)n_maps * tiles_y * tiles_x;
    const long long cap = 148ll * 32;
    tl::postprocess_bwd_kernel<<<(int)(n_tiles < cap ? n_tiles : cap), 256, 0, st>>>(a, tiles_y, tiles_x);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

}  // extern "C"

extern "C" {

namespace {
int dice_ce_args(tl::DiceCeArgs& a, const float* x, const float* t, int B, int C, int HW, void* ws) {
    if (!x || !t || !ws) return fail(TL_ERR_ARG, "null pointer");
    if (B <= 0 || C <= 0 || HW <= 0) return fail(TL_ERR_ARG, "bad shape [%d,%d,%d]", B, C, HW);
    if (C > tl::kDcMaxC) return fail(TL_ERR_ARG, "at most %d channels (got %d)", tl::kDcMaxC, C);
    if ((long long)B * C * HW >= (1ll << 40)) return fail(TL_ERR_ARG, "too large");
    a.x = x; a.t = t; a.B = B; a.C = C; a.HW = HW;
    a.tiles = (HW + tl::kDcThreads * tl::kDcPix - 1) / (tl::kDcThreads * tl::kDcPix);
    a.acc = static_cast<double*>(ws); a.loss_out = nullptr; a.grad_loss = nullptr; a.gx = nullptr;
    return TL_OK;
}
int dice_ce_grid(const tl::DiceCeArgs& a) {
    const long long jobs = (long long)a.B * a.tiles, cap = 148ll * 8;
    return (int)(jobs < cap ? jobs : cap);
}
}  // namespace

int tl_dice_ce_workspace_bytes(int B, int C, size_t* bytes) {
    if (!bytes || B <= 0 || C <= 0) return fail(TL_ERR_ARG, "bad arguments");
    *bytes = sizeof(double) * ((size_t)B * C * 3 + 1);
    return TL_OK;
}

int tl_dice_ce_forward(const float* logits, const float* target, int B, int C, int HW, void* ws, float* loss_out, void* stream) {
    tl::DiceCeArgs a;
    int rc = dice_ce_args(a, logits, target, B, C, HW, ws);
    if (rc != TL_OK) return rc;
    if (!loss_out) return fail(TL_ERR_ARG, "null pointer");
    a.loss_out = loss_out;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    TL_CUDA(cudaMemsetAsync(ws, 0, sizeof(double) * ((size_t)B * C * 3 + 1), st));
    tl::dice_ce_fwd_kernel<<<dice_ce_grid(a), tl::kDcThreads, 0, st>>>(a);
    TL_CUDA(cudaGetLastError());
    tl::dice_ce_finish_kernel<<<1, 256, 0, st>>>(a);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_dice_ce_backward(const float* grad_loss, const float* logits, const float* target, int B, int C, int HW,
                        const void* ws, float* grad_logits, void* stream) {
    tl::DiceCeArgs a;
    int rc = dice_ce_args(a, logits, target, B, C, HW, const_cast<void*>(ws));
    if (rc != TL_OK) return rc;
    if (!grad_logits) return fail(TL_ERR_ARG, "null pointer");
    a.grad_loss = grad_loss; a.gx = grad_logits;
    tl::dice_ce_bwd_kernel<<<dice_ce_grid(a), tl::kDcThreads, 0, static_cast<cudaStream_t>(stream)>>>(a);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

}  // extern "C"

// ---- Betti matching (tl_betti_*)
namespace {

constexpr int kBettiSlots = 148;  // CTAs of betti_kernel (one 1024-thread CTA per SM of a B200), each with its own tables

// [header 256 | counts [3][n] | recoff [n] | record arena | per-slot merge trees | per-slot node / edge tables]
//   header: [0] job counter (u32) | [8] arena head (u64) | [16] status (u32)
struct BettiLayout {
    size_t counts, recoff, arena, T, tabs, total;
    size_t t_stride, n_stride, e_stride, tab_stride;
    unsigned long long cap;
    int slots;
};
BettiLayout make_betti_layout(int n_maps, int H, int W, int dim) {
    BettiLayout B;
    memset(&B, 0, sizeof(B));
    size_t o = 256;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes); return at; };
    B.counts = take(sizeof(int32_t) * 3 * (size_t)n_maps);
    B.recoff = take(sizeof(uint32_t) * (size_t)n_maps);
    // a map's records: every interval of the prediction (matched or not) and every unmatched one of the target
    unsigned long long recs = (unsigned long long)n_maps * 2ull * (unsigned long long)max_pairs(H, W, dim);
    if (!opt(TL_OPT_WORST_CASE_WORKSPACE) && recs > (1ull << 28)) recs = 1ull << 28;  // 4 GiB of records
    if (recs > 0xFFFFFFFFull) recs = 0xFFFFFFFFull;
    B.cap = recs;
    B.arena = take(sizeof(int4) * (size_t)recs);
    B.slots = n_maps < kBettiSlots ? n_maps : kBettiSlots;
    const size_t nn = dim == 1 ? (size_t)H * W + 1 : (size_t)(H + 1) * (W + 1);
    const size_t ne = (size_t)H * (W + 1) + (size_t)(H + 1) * W;
    B.t_stride = align_up(sizeof(uint64_t) * nn) / sizeof(uint64_t);
    B.T = take(sizeof(uint64_t) * B.t_stride * B.slots);
    B.n_stride = align_up(sizeof(int32_t) * nn) / sizeof(int32_t);
    B.e_stride = align_up(sizeof(int32_t) * ne) / sizeof(int32_t);
    B.tab_stride = 6 * B.n_stride + 2 * B.e_stride;
    B.tabs = take(sizeof(int32_t) * B.tab_stride * B.slots);
    B.total = o;
    return B;
}

int betti_args(int n_maps, int H, int W, int dim, const void* ws, size_t ws_bytes, BettiLayout* B) {
    int rc = check_shape(n_maps, 1, H, W, dim);
    if (rc != TL_OK) return rc;
    if (!ws) return fail(TL_ERR_ARG, "null pointer");
    *B = make_betti_layout(n_maps, H, W, dim);
    if (ws_bytes < B->total) return fail(TL_ERR_ARG, "workspace %zu < %zu bytes (tl_betti_workspace_bytes)", ws_bytes, B->total);
    if (B->cap > 0x7FFFFFFFull) return fail(TL_ERR_ARG, "%d maps of %dx%d can hold more records than int32 offsets address", n_maps, H, W);
    return TL_OK;
}

// host copy of offsets [3][n_maps + 1]: each list starts at 0, never decreases and ends at its total
int check_host_offsets(const int32_t* host, int n_maps, const long long* totals) {
    static const char* what[3] = {"matched", "unmatched_pred", "unmatched_target"};
    for (int k = 0; k < 3; ++k) {
        const int32_t* h = host + (size_t)k * (n_maps + 1);
        if (h[0] != 0) return fail(TL_ERR_ARG, "%s offsets[0] = %d, not 0", what[k], h[0]);
        for (int i = 0; i < n_maps; ++i)
            if (h[i + 1] < h[i]) return fail(TL_ERR_ARG, "%s offsets decrease at map %d", what[k], i);
        if ((long long)h[n_maps] != totals[k]) return fail(TL_ERR_ARG, "%s count %lld disagrees with offsets[%d] = %d", what[k], totals[k], n_maps, h[n_maps]);
    }
    return TL_OK;
}

}  // namespace

extern "C" {

int tl_betti_workspace_bytes(int n_maps, int H, int W, int dim, size_t* bytes) {
    if (!bytes) return fail(TL_ERR_ARG, "bytes is null");
    int rc = check_shape(n_maps, 1, H, W, dim);
    if (rc != TL_OK) return rc;
    *bytes = make_betti_layout(n_maps, H, W, dim).total;
    return TL_OK;
}

int tl_betti_compute(const float* pred, const float* target, int n_maps, int H, int W, int dim, void* ws, size_t ws_bytes,
                     float* cost, int32_t* offsets, int32_t* status, void* stream) {
    BettiLayout B;
    int rc = betti_args(n_maps, H, W, dim, ws, ws_bytes, &B);
    if (rc != TL_OK) return rc;
    if (!pred || !target || !cost || !offsets) return fail(TL_ERR_ARG, "null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    TL_CUDA(cudaMemsetAsync(ws, 0, 256, st));  // job counter, arena head, status
    tl::BettiArgs a;
    a.pred = pred; a.target = target; a.n_maps = n_maps; a.H = H; a.W = W;
    a.job_counter = at<unsigned int>(ws, 0);
    a.head = at<unsigned long long>(ws, 8);
    a.cap = B.cap;
    a.arena = at<int4>(ws, B.arena);
    a.recoff = at<uint32_t>(ws, B.recoff);
    a.counts = at<int32_t>(ws, B.counts);
    a.cost = cost;
    a.status = at<unsigned int>(ws, 16);
    a.T = at<uint64_t>(ws, B.T); a.t_stride = B.t_stride;
    a.tabs = at<int32_t>(ws, B.tabs); a.tab_stride = B.tab_stride; a.n_stride = B.n_stride; a.e_stride = B.e_stride;
    if (dim == 1) tl::betti_kernel<1><<<B.slots, tl::kBmThreads, 0, st>>>(a);
    else tl::betti_kernel<0><<<B.slots, tl::kBmThreads, 0, st>>>(a);
    TL_CUDA(cudaGetLastError());
    for (int k = 0; k < 3; ++k) {
        tl::diagram_offsets_kernel<<<1, tl::kScanThreads, 0, st>>>(a.counts + (size_t)k * n_maps, n_maps, a.status,
                                                                    offsets + (size_t)k * (n_maps + 1), k == 2 ? status : nullptr);
        TL_CUDA(cudaGetLastError());
    }
    return TL_OK;
}

int tl_betti_gather(int n_maps, int H, int W, int dim, const void* ws, size_t ws_bytes, const int32_t* offsets,
                    const int32_t* host_offsets, long long M, long long Kp, long long Kt, int32_t* matched,
                    int32_t* unmatched_pred, int32_t* unmatched_target, void* stream) {
    BettiLayout B;
    int rc = betti_args(n_maps, H, W, dim, ws, ws_bytes, &B);
    if (rc != TL_OK) return rc;
    if (!offsets || !host_offsets) return fail(TL_ERR_ARG, "null pointer");
    if (M < 0 || Kp < 0 || Kt < 0 || (M > 0 && !matched) || (Kp > 0 && !unmatched_pred) || (Kt > 0 && !unmatched_target))
        return fail(TL_ERR_ARG, "null output buffer for %lld / %lld / %lld records", M, Kp, Kt);
    if (misaligned8(matched) || misaligned8(unmatched_pred) || misaligned8(unmatched_target))
        return fail(TL_ERR_ARG, "matched, unmatched_pred and unmatched_target must be 8-byte aligned");
    const long long totals[3] = {M, Kp, Kt};
    rc = check_host_offsets(host_offsets, n_maps, totals);
    if (rc != TL_OK) return rc;
    if (M + Kp + Kt == 0) return TL_OK;
    void* w = const_cast<void*>(ws);
    tl::betti_gather_kernel<<<n_maps < 1184 ? n_maps : 1184, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        at<int4>(w, B.arena), at<uint32_t>(w, B.recoff), n_maps, offsets, reinterpret_cast<int2*>(matched),
        reinterpret_cast<int2*>(unmatched_pred), reinterpret_cast<int2*>(unmatched_target));
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_betti_backward(const float* pred, const float* target, int n_maps, int H, int W, const int32_t* offsets,
                      const int32_t* matched, long long M, const int32_t* unmatched_pred, long long Kp,
                      const int32_t* unmatched_target, long long Kt, const float* grad_cost, float* grad_pred,
                      float* grad_target, void* stream) {
    if (n_maps <= 0 || H <= 0 || W <= 0 || (long long)H * W >= 0x7FFFFFF0LL) return fail(TL_ERR_ARG, "bad shape [%d,%d,%d]", n_maps, H, W);
    if (!pred || !target || !offsets || !grad_cost || !grad_pred) return fail(TL_ERR_ARG, "null pointer");
    if (M < 0 || Kp < 0 || Kt < 0 || (M > 0 && !matched) || (Kp > 0 && !unmatched_pred) || (Kt > 0 && !unmatched_target))
        return fail(TL_ERR_ARG, "null record buffer for %lld / %lld / %lld records", M, Kp, Kt);
    if (misaligned8(matched) || misaligned8(unmatched_pred) || misaligned8(unmatched_target))
        return fail(TL_ERR_ARG, "matched, unmatched_pred and unmatched_target must be 8-byte aligned");
    tl::BettiBwdArgs a;
    a.pred = pred; a.target = target; a.n_maps = n_maps; a.N = H * W; a.offsets = offsets;
    a.matched = reinterpret_cast<const int2*>(matched);
    a.up = reinterpret_cast<const int2*>(unmatched_pred); a.ut = reinterpret_cast<const int2*>(unmatched_target);
    a.grad_cost = grad_cost; a.grad_pred = grad_pred; a.grad_target = grad_target;
    tl::betti_backward_kernel<<<n_maps < 1184 ? n_maps : 1184, 512, 0, static_cast<cudaStream_t>(stream)>>>(a);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

}  // extern "C"

// ---- topological prior (tl_prior_*)
namespace {

// STATE: the pairs layout's state part (header, bookkeeping, the sorted arena), then the per-map threshold keys;
// SCRATCH: the pairs layout's scratch part (its sort-key array holds the records' p bits during the forward)
struct PriorLayout { PairsLayout P; size_t thr, state_bytes, scratch_bytes; };
PriorLayout make_prior_layout(int n_maps, int H, int W, int dim) {
    PriorLayout R;
    R.P = make_pairs_layout(n_maps, H, W, dim);
    R.thr = R.P.state_bytes;  // 256-byte aligned
    R.state_bytes = R.thr + align_up(sizeof(uint64_t) * (size_t)n_maps);
    R.scratch_bytes = R.P.L.total;
    return R;
}

int prior_args(int n_maps, int H, int W, int dim, const float* maps, const void* state, size_t state_bytes, PriorLayout* R) {
    int rc = check_shape(n_maps, 1, H, W, dim);
    if (rc != TL_OK) return rc;
    if (!maps || !state) return fail(TL_ERR_ARG, "null pointer");
    *R = make_prior_layout(n_maps, H, W, dim);
    if (state_bytes < R->state_bytes) return fail(TL_ERR_ARG, "state %zu < %zu bytes (tl_prior_workspace_bytes)", state_bytes, R->state_bytes);
    return TL_OK;
}

}  // namespace

extern "C" {

int tl_prior_workspace_bytes(int n_maps, int H, int W, int dim, size_t* state_bytes, size_t* scratch_bytes) {
    if (!state_bytes || !scratch_bytes) return fail(TL_ERR_ARG, "null pointer");
    int rc = check_shape(n_maps, 1, H, W, dim);
    if (rc != TL_OK) return rc;
    const PriorLayout R = make_prior_layout(n_maps, H, W, dim);
    *state_bytes = R.state_bytes;
    *scratch_bytes = R.scratch_bytes;
    return TL_OK;
}

int tl_prior_forward(const float* maps, int n_maps, int H, int W, int dim, const int32_t* betti, void* state,
                     size_t state_bytes, void* scratch, size_t scratch_bytes, float* cost, void* stream) {
    PriorLayout R;
    int rc = prior_args(n_maps, H, W, dim, maps, state, state_bytes, &R);
    if (rc != TL_OK) return rc;
    if (!betti || !scratch || !cost) return fail(TL_ERR_ARG, "null pointer");
    if (scratch_bytes < R.scratch_bytes) return fail(TL_ERR_ARG, "scratch %zu < %zu bytes (tl_prior_workspace_bytes)", scratch_bytes, R.scratch_bytes);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    tl::PairStore ps;
    rc = sorted_pairs(maps, n_maps, H, W, dim, state, scratch, R.P, st, &ps);
    if (rc != TL_OK) return rc;
    tl::PriorArgs a;
    a.arena = ps.arena; a.offs = ps.offs[0]; a.counts = ps.counts[0];
    a.maps = maps; a.N = (long long)H * W; a.n_maps = n_maps;
    a.betti = betti; a.status = ps.status;
    a.pbits = reinterpret_cast<uint32_t*>(ps.skeys);  // the sort is done with its keys; half of each 8-byte slot is used
    a.thr = at<uint64_t>(state, R.thr);
    a.cost = cost;
    tl::prior_cost_kernel<<<n_maps < 1184 ? n_maps : 1184, tl::kPriorThreads, 0, st>>>(a);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

int tl_prior_backward(const float* maps, int n_maps, int H, int W, int dim, const void* state, size_t state_bytes,
                      const float* grad_cost, float* grad_maps, void* stream) {
    PriorLayout R;
    int rc = prior_args(n_maps, H, W, dim, maps, state, state_bytes, &R);
    if (rc != TL_OK) return rc;
    if (!grad_cost || !grad_maps) return fail(TL_ERR_ARG, "null pointer");
    void* w = const_cast<void*>(state);
    tl::PriorBwdArgs a;
    a.arena = at<tl::PairRec>(w, R.P.S.arena); a.offs = at<uint32_t>(w, R.P.S.offs[0]); a.counts = at<int32_t>(w, R.P.S.counts[0]);
    a.maps = maps; a.N = H * W; a.n_maps = n_maps;
    a.thr = at<uint64_t>(w, R.thr);
    a.status = at<unsigned int>(w, 16);
    a.grad_cost = grad_cost; a.grad_maps = grad_maps;
    tl::prior_backward_kernel<<<n_maps < 1184 ? n_maps : 1184, 512, 0, static_cast<cudaStream_t>(stream)>>>(a);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

}  // extern "C"

// ---- exact Euclidean distance transform (tl_edt) and the Hausdorff distance-transform loss (tl_hausdorff_dt_*)
namespace {

int edt_shape(int n_maps, int H, int W) {
    if (n_maps <= 0 || H < 1 || W < 1 || H > tl::kEdtMaxDim || W > tl::kEdtMaxDim)
        return fail(TL_ERR_ARG, "bad shape [%d,%d,%d] (n_maps > 0, H and W in [1, %d])", n_maps, H, W, tl::kEdtMaxDim);
    return TL_OK;
}

// STATE: D = F(P)^alpha + F(T)^alpha, fp32 per pixel (the backward reads it); SCRATCH: the row pass's h0 / h1 of one
// mask, a uint2 per pixel (P, then T)
size_t edt_pixels(int n_maps, int H, int W) { return (size_t)n_maps * H * W; }

int edt_grid(long long work, int per_block) {
    const long long b = (work + per_block - 1) / per_block;
    return (int)(b < (1ll << 20) ? b : (1ll << 20));
}

template <class Src, int NL>
int edt_rows(Src src, int n_maps, int H, int W, uint32_t* h, cudaStream_t st) {
    const long long rows = (long long)n_maps * H;
    tl::edt_row_kernel<Src, NL><<<edt_grid(rows, tl::kEdtRowWarps), tl::kEdtRowWarps * 32, 0, st>>>(src, rows, W, h);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

template <int Mode, bool kSp = false>
int edt_cols(const tl::EdtColArgs& a, cudaStream_t st) {
    tl::edt_col_kernel<Mode, kSp><<<a.n_maps < (1 << 20) ? a.n_maps : (1 << 20), tl::kEdtColThreads, 0, st>>>(a);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

// tl_edt and tl_edt_spaced (kSp: spacing is a device [n][2] array, checked non-null by the caller)
template <bool kSp>
int edt_field(const uint8_t* mask, int n_maps, int H, int W, const double* spacing, void* ws, size_t ws_bytes,
              float* out, void* stream) {
    int rc = edt_shape(n_maps, H, W);
    if (rc != TL_OK) return rc;
    if (!mask || !ws || !out) return fail(TL_ERR_ARG, "null pointer");
    if (reinterpret_cast<uintptr_t>(ws) & 3) return fail(TL_ERR_ARG, "workspace must be 4-byte aligned");
    const size_t need = align_up(sizeof(uint32_t) * edt_pixels(n_maps, H, W));
    if (ws_bytes < need) return fail(TL_ERR_ARG, "workspace %zu < %zu bytes (tl_edt_workspace_bytes)", ws_bytes, need);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint32_t* h = static_cast<uint32_t*>(ws);
    rc = edt_rows<tl::EdtMaskSrc, 1>(tl::EdtMaskSrc{mask}, n_maps, H, W, h, st);
    if (rc != TL_OK) return rc;
    tl::EdtColArgs a = {};
    a.h = h; a.n_maps = n_maps; a.H = H; a.W = W; a.field = out; a.spacing = spacing;
    return edt_cols<tl::kEdtField, kSp>(a, st);
}

// tl_hausdorff_dt_forward and its _spaced form
template <bool kSp>
int hausdorff_dt_forward(const float* logits, const float* target, int n_maps, int H, int W, double alpha,
                         const double* spacing, void* state, size_t state_bytes, void* scratch, size_t scratch_bytes,
                         float* cost, void* stream) {
    int rc = edt_shape(n_maps, H, W);
    if (rc != TL_OK) return rc;
    if (!logits || !target || !state || !scratch || !cost) return fail(TL_ERR_ARG, "null pointer");
    if (!(alpha > 0.0) || !(alpha < HUGE_VAL)) return fail(TL_ERR_ARG, "alpha must be finite and positive, got %g", alpha);
    if ((reinterpret_cast<uintptr_t>(state) & 3) || (reinterpret_cast<uintptr_t>(scratch) & 7))
        return fail(TL_ERR_ARG, "state must be 4-byte and scratch 8-byte aligned");
    const size_t ns = align_up(sizeof(float) * edt_pixels(n_maps, H, W)), nc = align_up(sizeof(uint2) * edt_pixels(n_maps, H, W));
    if (state_bytes < ns) return fail(TL_ERR_ARG, "state %zu < %zu bytes (tl_hausdorff_dt_workspace_bytes)", state_bytes, ns);
    if (scratch_bytes < nc) return fail(TL_ERR_ARG, "scratch %zu < %zu bytes (tl_hausdorff_dt_workspace_bytes)", scratch_bytes, nc);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    tl::EdtColArgs a = {};
    a.h = static_cast<uint32_t*>(scratch); a.n_maps = n_maps; a.H = H; a.W = W;
    a.sp = static_cast<int32_t*>(state); a.D = static_cast<float*>(state);
    a.x = logits; a.t = target; a.half_alpha = 0.5 * alpha; a.cost = cost; a.spacing = spacing;
    rc = edt_rows<tl::EdtLogitSrc, 2>(tl::EdtLogitSrc{logits}, n_maps, H, W, a.h, st);
    if (rc == TL_OK) rc = edt_cols<tl::kEdtPred, kSp>(a, st);
    if (rc == TL_OK) rc = edt_rows<tl::EdtTargetSrc, 2>(tl::EdtTargetSrc{target}, n_maps, H, W, a.h, st);
    if (rc == TL_OK) rc = edt_cols<tl::kEdtTarget, kSp>(a, st);
    return rc;
}

}  // namespace

extern "C" {

int tl_edt_workspace_bytes(int n_maps, int H, int W, size_t* bytes) {
    if (!bytes) return fail(TL_ERR_ARG, "null pointer");
    int rc = edt_shape(n_maps, H, W);
    if (rc != TL_OK) return rc;
    *bytes = align_up(sizeof(uint32_t) * edt_pixels(n_maps, H, W));
    return TL_OK;
}

int tl_edt(const uint8_t* mask, int n_maps, int H, int W, void* ws, size_t ws_bytes, float* out, void* stream) {
    return edt_field<false>(mask, n_maps, H, W, nullptr, ws, ws_bytes, out, stream);
}

int tl_edt_spaced(const uint8_t* mask, int n_maps, int H, int W, const double* spacing, void* ws, size_t ws_bytes,
                  float* out, void* stream) {
    if (!spacing) return fail(TL_ERR_ARG, "null pointer");
    if (reinterpret_cast<uintptr_t>(spacing) & 7) return fail(TL_ERR_ARG, "spacing must be 8-byte aligned");
    return edt_field<true>(mask, n_maps, H, W, spacing, ws, ws_bytes, out, stream);
}

int tl_hausdorff_dt_workspace_bytes(int n_maps, int H, int W, size_t* state_bytes, size_t* scratch_bytes) {
    if (!state_bytes || !scratch_bytes) return fail(TL_ERR_ARG, "null pointer");
    int rc = edt_shape(n_maps, H, W);
    if (rc != TL_OK) return rc;
    *state_bytes = align_up(sizeof(float) * edt_pixels(n_maps, H, W));
    *scratch_bytes = align_up(sizeof(uint2) * edt_pixels(n_maps, H, W));
    return TL_OK;
}

int tl_hausdorff_dt_forward(const float* logits, const float* target, int n_maps, int H, int W, double alpha,
                            void* state, size_t state_bytes, void* scratch, size_t scratch_bytes, float* cost,
                            void* stream) {
    return hausdorff_dt_forward<false>(logits, target, n_maps, H, W, alpha, nullptr, state, state_bytes, scratch,
                                       scratch_bytes, cost, stream);
}

int tl_hausdorff_dt_forward_spaced(const float* logits, const float* target, int n_maps, int H, int W, double alpha,
                                   const double* spacing, void* state, size_t state_bytes, void* scratch,
                                   size_t scratch_bytes, float* cost, void* stream) {
    if (!spacing) return fail(TL_ERR_ARG, "null pointer");
    if (reinterpret_cast<uintptr_t>(spacing) & 7) return fail(TL_ERR_ARG, "spacing must be 8-byte aligned");
    return hausdorff_dt_forward<true>(logits, target, n_maps, H, W, alpha, spacing, state, state_bytes, scratch,
                                      scratch_bytes, cost, stream);
}

int tl_hausdorff_dt_backward(const float* logits, const float* target, int n_maps, int H, int W, const void* state,
                             size_t state_bytes, const float* grad_cost, float* grad_logits, void* stream) {
    int rc = edt_shape(n_maps, H, W);
    if (rc != TL_OK) return rc;
    if (!logits || !target || !state || !grad_cost || !grad_logits) return fail(TL_ERR_ARG, "null pointer");
    if (reinterpret_cast<uintptr_t>(state) & 3) return fail(TL_ERR_ARG, "state must be 4-byte aligned");
    const size_t ns = align_up(sizeof(float) * edt_pixels(n_maps, H, W));
    if (state_bytes < ns) return fail(TL_ERR_ARG, "state %zu < %zu bytes (tl_hausdorff_dt_workspace_bytes)", state_bytes, ns);
    const long long N = (long long)H * W;
    tl::hausdorff_dt_backward_kernel<<<edt_grid((long long)n_maps * ((N + 1023) / 1024), 1), 256, 0,
                                       static_cast<cudaStream_t>(stream)>>>(
        logits, target, static_cast<const float*>(state), grad_cost, n_maps, N, grad_logits);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

}  // extern "C"

// ---- surface-distance metrics (tl_surface_*)
namespace {

// the row pass's h of both surfaces, then the keys of both directions (uint32 per pixel each), then [4][n] stats
struct SurfLayout {
    size_t keys, stats, total;
};

SurfLayout surface_layout(int n_maps, int H, int W) {
    SurfLayout L;
    const size_t px = edt_pixels(n_maps, H, W);
    L.keys = align_up(sizeof(uint32_t) * 2 * px);
    L.stats = L.keys + align_up(sizeof(uint32_t) * 2 * px);
    L.total = L.stats + align_up(sizeof(uint32_t) * 4 * (size_t)n_maps);
    return L;
}

template <bool kSp>
int surface_distances(const uint8_t* pred, const uint8_t* target, int n_maps, int H, int W, const double* spacing,
                      double percentile, double tolerance, void* ws, size_t ws_bytes, float* out, void* stream) {
    int rc = edt_shape(n_maps, H, W);
    if (rc != TL_OK) return rc;
    if (!pred || !target || !ws || !out) return fail(TL_ERR_ARG, "null pointer");
    if (!(percentile >= 0.0 && percentile <= 100.0)) return fail(TL_ERR_ARG, "percentile must be in [0, 100], got %g", percentile);
    if (!(tolerance >= 0.0 && tolerance < HUGE_VAL)) return fail(TL_ERR_ARG, "tolerance must be finite and >= 0, got %g", tolerance);
    if (reinterpret_cast<uintptr_t>(ws) & 3) return fail(TL_ERR_ARG, "workspace must be 4-byte aligned");
    const SurfLayout L = surface_layout(n_maps, H, W);
    if (ws_bytes < L.total) return fail(TL_ERR_ARG, "workspace %zu < %zu bytes (tl_surface_workspace_bytes)", ws_bytes, L.total);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    char* base = static_cast<char*>(ws);
    tl::SurfArgs a = {};
    a.h = reinterpret_cast<uint32_t*>(base);
    a.keys = reinterpret_cast<uint32_t*>(base + L.keys);
    a.stats = reinterpret_cast<uint32_t*>(base + L.stats);
    a.n_maps = n_maps; a.H = H; a.W = W;
    a.tol = tolerance; a.qq = percentile / 100.0; a.out = out; a.spacing = spacing;
    rc = edt_rows<tl::SurfSrc, 1>(tl::SurfSrc{pred, H, W}, n_maps, H, W, a.h, st);
    if (rc == TL_OK) rc = edt_rows<tl::SurfSrc, 1>(tl::SurfSrc{target, H, W}, n_maps, H, W, a.h + edt_pixels(n_maps, H, W), st);
    if (rc != TL_OK) return rc;
    const int grid = n_maps < (1 << 20) ? n_maps : (1 << 20);
    tl::surface_col_kernel<kSp><<<grid, tl::kEdtColThreads, 0, st>>>(a);
    TL_CUDA(cudaGetLastError());
    tl::surface_select_kernel<kSp><<<grid, tl::kSurfSelThreads, 0, st>>>(a);
    TL_CUDA(cudaGetLastError());
    return TL_OK;
}

}  // namespace

extern "C" {

int tl_surface_workspace_bytes(int n_maps, int H, int W, size_t* bytes) {
    if (!bytes) return fail(TL_ERR_ARG, "null pointer");
    int rc = edt_shape(n_maps, H, W);
    if (rc != TL_OK) return rc;
    *bytes = surface_layout(n_maps, H, W).total;
    return TL_OK;
}

int tl_surface_distances(const uint8_t* pred, const uint8_t* target, int n_maps, int H, int W, double percentile,
                         double tolerance, void* ws, size_t ws_bytes, float* out, void* stream) {
    return surface_distances<false>(pred, target, n_maps, H, W, nullptr, percentile, tolerance, ws, ws_bytes, out, stream);
}

int tl_surface_distances_spaced(const uint8_t* pred, const uint8_t* target, int n_maps, int H, int W,
                                const double* spacing, double percentile, double tolerance, void* ws, size_t ws_bytes,
                                float* out, void* stream) {
    if (!spacing) return fail(TL_ERR_ARG, "null pointer");
    if (reinterpret_cast<uintptr_t>(spacing) & 7) return fail(TL_ERR_ARG, "spacing must be 8-byte aligned");
    return surface_distances<true>(pred, target, n_maps, H, W, spacing, percentile, tolerance, ws, ws_bytes, out, stream);
}

}  // extern "C"
