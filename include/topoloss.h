/*
 * topoloss.h -- C ABI of libtopoloss.so: the B200 (sm_100a) topological-loss hot path.
 *
 * This is the drop-in boundary for the one path the library replaces:
 *
 *   topo_loss(pred_obj, true_obj, lamda, interp, feat_d, loss_q, loss_r)
 *       /root/reference/octsam/models/topological_loss.py:11-96
 *   called from the SAM fine-tuning step at
 *       /root/reference/octsam/models/training_utils.py:64 (train) and :375 (validation)
 *   and differentiated by  train_loss.backward()  (training_utils.py:66).
 *
 * The reference has no FFI of its own (it is a Python callable over torch_topological ->
 * gudhi / POT); the entry points below are what a ctypes binding of that callable binds:
 * INTEGRATION.md shows the stub.  Plain pointers and sizes only, no torch types.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its comment says host;
 *   - the caller owns every buffer, including the two workspaces (sizes from
 *     tl_workspace_bytes): STATE, which tl_forward fills and tl_backward reads, and SCRATCH,
 *     which is only live inside one call and may be shared by every call enqueued on the same
 *     stream; the library never allocates or frees device memory and keeps no device state.
 *     The only host state is process-wide: the options below and the timing aid;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no entry point
 *     synchronises the host with the device;
 *   - every function returns TL_OK (0) or a negative TL_ERR_* code; tl_last_error()
 *     returns a thread-local, human-readable message for the last failure;
 *   - maps are [B, C, H, W] fp32, contiguous (NCHW): one (image, class) map is one
 *     contiguous H*W segment.  Pixels are the top-dimensional cells of the cubical
 *     complex (gudhi T-construction), sublevel filtration, as CubicalComplex(dim=2,
 *     superlevel=False) at topological_loss.py:55-58.
 *   - persistence pairs are (creator pixel, destroyer pixel) flat C-order indices r*W+c.
 *   - H and W are the map's geometry AS gudhi SEES IT: H rows of W pixels, W the fastest axis.  For
 *     square maps that is the tensor's own shape.  For H != W, torch_topological hands gudhi
 *     `dimensions=x.shape` un-reversed while gudhi's first dimension is the fastest one, so the
 *     reference computes the persistence of the SAME flat buffer read as W rows of H pixels: a
 *     caller that wants the reference's result for a [.., h, w] tensor passes H = w, W = h (flat
 *     indices, and therefore the gradient layout, are unchanged).  The Python shim does this.
 *   - no CPU fallback exists: without a CUDA device every compute entry point fails.
 */
#ifndef TOPOLOSS_H_
#define TOPOLOSS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TL_OK 0
#define TL_ERR_ARG (-1)       /* bad argument (shape, feat_d, null pointer, ...) */
#define TL_ERR_WORKSPACE (-2) /* workspace too small */
#define TL_ERR_CUDA (-3)      /* a CUDA runtime call failed; see tl_last_error() */

#define TL_ABI_VERSION 4

/* ABI version of the loaded library (TL_ABI_VERSION it was built with). */
int tl_version(void);

/* Thread-local message for the last error returned on this thread ("" if none). */
const char* tl_last_error(void);

/*
 * Process-wide options.  Initial values are read from the environment ONCE, when the library is
 * loaded (TL_FORCE_GLOBAL, TL_PROFILE, TL_NO_BINARY, TL_WORST_CASE_WORKSPACE, TL_NO_FUSED_MATCH, TL_NO_FUSED_GRAD = "1"); tl_set_option
 * changes them afterwards.  FORCE_GLOBAL_KERNEL and WORST_CASE_WORKSPACE change the workspace layout:
 * use the same setting for tl_workspace_bytes and the calls that consume its sizes.
 */
#define TL_OPT_FORCE_GLOBAL_KERNEL 0  /* tests: every shape through the global-memory persistence kernel */
#define TL_OPT_PROFILE 1              /* accumulate per-phase cycle counters (tl_debug_profile) */
#define TL_OPT_NO_BINARY_PATH 2       /* measurement: two-valued maps through the generic path */
#define TL_OPT_WORST_CASE_WORKSPACE 3 /* size every table for the worst case: no input can overflow */
#define TL_OPT_NO_FUSED_MATCH 4       /* measurement: matching in a launch of its own instead of the persistence kernel's tail */
#define TL_OPT_NO_FUSED_GRAD 5        /* measurement: tl_forward_backward writes the gradient in a launch of its own */
#define TL_OPT_LIST_MODE 6            /* measurement (env TL_LIST_MODE, an integer): L2 treatment of the per-CTA crossing-edge list of
                                         single-band maps.  bit 0: discard the list's L2 lines once the merge has consumed them (no
                                         write-back of scratch data); bit 1: store the list with an evict-last policy; bit 2: read
                                         the maps without the evict-last hint */
#define TL_OPT_COUNT_ 7
int tl_set_option(int which, int value);
int tl_get_option(int which);

/*
 * Bytes of device memory tl_forward / tl_backward need for maps of this shape.  feat_d in {0, 1} is
 * the homology dimension that will be used (batch_iter(..., dim=feat_d), topological_loss.py:68-75).
 *   *state_bytes    header + per-map bookkeeping + the PAIR ARENA: one pool of (creator, destroyer,
 *                   birth, death, matched point) records shared by all maps, carved with a device
 *                   counter.  The returned size holds max(H*W/5 + 64, 8192) pairs per map, both sets together
 *                   (a noise-like prediction produces ~H*W/5, segmentation ground truth a handful; maps
 *                   up to 128 x 128 thereby get the combinatorial maximum); any LARGER buffer is used in full.  With TL_OPT_WORST_CASE_WORKSPACE it holds the
 *                   combinatorial maximum (H*W/2 + 2 per map and set).
 *   *scratch_bytes  per-CTA tables of the persistence kernels (independent of B).
 * Both are host pointers.  If a pathological input exhausts the arena (or, on maps of more than
 * 65536 pixels with the typical-size tables, the basin tables) nothing is written out of bounds: a
 * status bit is set, the loss becomes NaN and tl_status reports it.
 */
int tl_workspace_bytes(int B, int C, int H, int W, int feat_d, size_t* state_bytes, size_t* scratch_bytes);

#define TL_STATUS_ARENA 1     /* pair arena exhausted */
#define TL_STATUS_BASINS 2    /* basin tables exhausted (multi-band maps, typical-size workspace) */
#define TL_STATUS_NONFINITE 4 /* a map holds a NaN */
/* Host copy of the status word of the last tl_forward that used `state` (0 = fine).  Synchronises `stream`. */
int tl_status(const void* state, int* host_status, void* stream);

/*
 * Forward pass of topo_loss for interp == 0 (topological_loss.py:55-96):
 *   per (b, c) map: cubical persistence pairs of pred and truth in dimension feat_d
 *                   (CubicalComplex.forward, :62-63; essential H0 class paired with argmax),
 *   per map:        exact q-Wasserstein matching cost with L-inf ground metric
 *                   (WassersteinDistance(q=loss_q), :78-82),
 *   per image:      W_b = (sum_c cost_{b,c})^(1/q),
 *   loss = lamda / B_global * sum_b W_b                       (:85, :96)
 *          [+ lamda / (B_global*C) * sum_{b,c} sum_pairs |d-b|^q   if loss_r (:88-94)].
 * B_global is the batch size the mean runs over; pass B (or 0) on one GPU, the global
 * batch when the batch axis is sharded over ranks (the caller then all-reduces loss_out).
 * loss_out: one fp32 on the device.  `state` keeps what tl_backward needs.
 */
int tl_forward(const float* pred, const float* truth, int B, int C, int H, int W,
               int feat_d, float q, float lamda, int loss_r, int B_global,
               void* state, size_t state_bytes, void* scratch, size_t scratch_bytes,
               float* loss_out, void* stream);

/*
 * Backward pass (the autograd graph of training_utils.py:66 restricted to this loss):
 * grad_pred[B,C,H,W] = grad_loss * d loss / d pred, fully overwritten (zeros included).
 * grad_loss: one fp32 on the device (upstream gradient), or NULL for 1.0.
 * `state` must be the buffer a tl_forward call filled; shape, feat_d, q, lamda, loss_r and
 * B_global must be the values given to that call (the library keeps no state between calls).
 * An image whose summed cost S_b is exactly 0 gets NaN on all its critical pixels, as the
 * reference's autograd does (0 * inf through pow(1/q)).
 */
int tl_backward(const float* grad_loss, const void* state, size_t state_bytes,
                int B, int C, int H, int W, int feat_d, float q, float lamda, int loss_r,
                int B_global, float* grad_pred, void* stream);

/*
 * tl_forward and tl_backward (upstream gradient 1.0) as ONE call: what `loss = topo_loss(...); loss.backward()`
 * at training_utils.py:64-66 amounts to.  Same arguments and results as the two calls; grad_pred[B,C,H,W] is fully
 * overwritten.  The gradient of an image is written in the tail of the persistence launch as soon as its C maps
 * are matched, by SMs that have run out of persistence work, instead of in a launch of its own.  Scale the
 * result with tl_scale_gradient when the upstream gradient is not 1.
 */
int tl_forward_backward(const float* pred, const float* truth, int B, int C, int H, int W,
                        int feat_d, float q, float lamda, int loss_r, int B_global,
                        void* state, size_t state_bytes, void* scratch, size_t scratch_bytes,
                        float* loss_out, float* grad_pred, void* stream);

/*
 * grad_pred[0..n) *= *grad_loss (one fp32 on the device; NULL = 1.0).  The kernel returns without touching
 * grad_pred when the value is exactly 1.0, the case of a plain `loss.backward()`.
 */
int tl_scale_gradient(const float* grad_loss, float* grad_pred, long long n, void* stream);

/*
 * Ground-truth masks that crossed PCIe bit-packed: maps[i] = bit i of `bits` as 0.0f / 1.0f, numpy.packbits
 * order (pixel 0 is bit 7 of byte 0).  n_pixels must be a multiple of 8.  The reference builds the masks on the
 * CPU as {0.0, 1.0} arrays (training_utils.py:398, :413, :432); packed they are 1/32 of the fp32 bytes.
 */
int tl_unpack_mask_bits(const uint8_t* bits, float* maps, long long n_pixels, void* stream);

/*
 * Inner boundary for parity tests: CubicalComplex.forward on n_maps independent HxW maps
 * (torch_topological CubicalComplex._forward -> gudhi persistence +
 * cofaces_of_persistence_pairs).  Writes, per map, up to `cap` pairs
 * (creator, destroyer) of homology dimension `dim` into pairs[map][k][2], sorted in
 * gudhi's emission order (filtration order of the death cell; essential H0 class last),
 * and the count into counts[map].  A map with more than `cap` pairs reports its true count
 * and writes only the first `cap`.  `ws`: one buffer of tl_pairs_workspace_bytes bytes.
 */
int tl_pairs_workspace_bytes(int n_maps, int H, int W, int dim, size_t* bytes);
int tl_persistence_pairs(const float* maps, int n_maps, int H, int W, int dim,
                         void* ws, size_t ws_bytes,
                         int32_t* pairs, int cap, int32_t* counts, void* stream);

/* Largest number of pairs one HxW map can produce in dimension dim (buffer sizing). */
int tl_max_pairs(int H, int W, int dim);

/*
 * Inner boundary for parity tests: WassersteinDistance cost of one channel, batched.
 * Diagram k of set 1 is rows off1[k]..off1[k+1]-1 of D1 ([rows][2] fp32 (birth, death)),
 * likewise D2/off2 (off arrays have n_diag+1 int32 entries, device).  Writes
 * cost[k] (fp64, the emd2 value before the 1/q root) and match1[row] = row index inside
 * diagram k of D2 that D1's row is matched to, or -1 for the diagonal.
 */
int tl_wasserstein(const float* D1, const int32_t* off1, const float* D2, const int32_t* off2,
                   int n_diag, int max_rows1, int max_rows2, float q,
                   void* ws, size_t ws_bytes, double* cost, int32_t* match1, void* stream);

/*
 * Debug aid, not on the hot path: host copy of the 8 per-phase cycle counters the persistence
 * kernel accumulates into the state buffer while TL_OPT_PROFILE is set.
 * Synchronises the device.  host_out8: 8 x uint64 on the host.
 */
int tl_debug_profile(const void* state, unsigned long long* host_out8);
/*
 * Debug aid: per-SM timeline of the tail of the last persistence launch that used `scratch` while TL_OPT_PROFILE
 * was set: 11 x uint64 per slot (ns of %globaltimer: persistence jobs done, exit; ns spent in matching / gradient
 * jobs; matching / gradient jobs run; cycles of the gradient jobs in tile zeroing / scatter / stream-out / record wait / barrier).  Returns the number of slots written (<= max_slots).  Synchronises the device.
 */
int tl_debug_tail_profile(const void* scratch, int H, int W, int feat_d, unsigned long long* host_out, int max_slots);

/*
 * Measurement aid for bench.py's roofline: while enabled (process-wide, mutex-guarded: the backward
 * runs on autograd's thread), tl_forward and tl_backward bracket their kernels with
 * cudaEventRecord on the caller's stream (the stream the kernels are launched on).
 * tl_timing_read synchronises those events and returns, on the host, the summed milliseconds of
 * the 6 stages [persistence, (unused), matching, loss, (unused), gradient fill + scatter] over the
 * calls since the last enable/read (at most 128), and the number of forward / backward calls in
 * n_calls[0..1].
 */
int tl_timing_enable(int on);
int tl_timing_read(float* ms_sum6, int* n_calls);

/*
 * F1 (SURVEY.md 8f), the step in front of the path at the reference call site
 *   topo_loss(torch.sigmoid(masks.float()), gt_masks.float(), 0.1, feat_d=1, interp=50)
 *       /root/reference/octsam/models/training_utils.py:64
 * i.e. torch.sigmoid followed by F.interpolate(size=(interp, interp), mode="bilinear",
 * align_corners=True) of /root/reference/octsam/models/topological_loss.py:33-46, fused:
 *   out[m, oy, ox] = bilinear_{align_corners}( apply_sigmoid ? sigmoid(in[m]) : in[m] )(oy, ox)
 * in: [n_maps][H][W] fp32 (logits when apply_sigmoid, e.g. the mask decoder output; plain maps
 * otherwise, e.g. ground truth), out: [n_maps][S][S].  Only the <= 4 S^2 source pixels an output
 * needs are read and passed through the sigmoid.
 */
int tl_resample_forward(const float* in, int n_maps, int H, int W, int S, int apply_sigmoid,
                        float* out, void* stream);

/*
 * Backward of tl_resample_forward: grad_in[n_maps][H][W] (16-byte aligned) is fully overwritten
 * with sum over outputs of weight * grad_out * (apply_sigmoid ? s(1-s) : 1); `in` are the forward inputs.
 */
int tl_resample_backward(const float* grad_out, const float* in, int n_maps, int H, int W, int S,
                         int apply_sigmoid, float* grad_in, void* stream);

/*
 * F3 (SURVEY.md 8f): SAM post-processing of the mask decoder output, fused into one gather:
 *   m   = F.interpolate(pred_masks.squeeze(2), (T, T), mode="bilinear", align_corners=False)   T = 1024
 *   m   = m[..., :rh, :rw]                                                  (reshaped_input_sizes)
 *   out = F.interpolate(m, (oh, ow), mode="bilinear", align_corners=False)  (original_sizes)
 *       /root/reference/octsam/models/training_utils.py:57-59
 * in: [n_maps][Hs][Ws] fp32, out: [n_maps][oh][ow].  The T x T intermediate is never materialised.
 */
int tl_postprocess_forward(const float* in, int n_maps, int Hs, int Ws, int T, int rh, int rw,
                           int oh, int ow, float* out, void* stream);

/* Backward of tl_postprocess_forward: grad_in[n_maps][Hs][Ws] (16-byte aligned) fully overwritten. */
int tl_postprocess_backward(const float* grad_out, int n_maps, int Hs, int Ws, int T, int rh, int rw,
                            int oh, int ow, float* grad_in, void* stream);

/*
 * F2 (SURVEY.md 8f): the sibling loss of the reference training step,
 *   seg_loss = monai.losses.DiceCELoss(sigmoid=True)     /root/reference/octsam/models/training_utils.py:32
 *   train_loss = seg_loss(masks, gt_masks)               training_utils.py:62
 * (monai 1.3.0, environment.yml:224: mean over (b, c) of 1 - (2 sum s t + 1e-5) / (sum s + sum t + 1e-5) with
 * s = sigmoid(logits), plus torch.nn.CrossEntropyLoss over the channel axis with the targets as class
 * probabilities) as one read of the two [B][C][HW] fp32 tensors per pass.  `ws`: tl_dice_ce_workspace_bytes
 * bytes, filled by the forward and read by the backward; loss_out: one fp32 on the device; grad_loss: one
 * fp32 on the device or NULL for 1.0; grad_logits [B][C][HW] is fully overwritten.  At most 64 channels.
 */
int tl_dice_ce_workspace_bytes(int B, int C, size_t* bytes);
int tl_dice_ce_forward(const float* logits, const float* target, int B, int C, int HW, void* ws,
                       float* loss_out, void* stream);
int tl_dice_ce_backward(const float* grad_loss, const float* logits, const float* target, int B, int C, int HW,
                        const void* ws, float* grad_logits, void* stream);

/* Bytes of workspace tl_wasserstein needs. */
int tl_wasserstein_workspace_bytes(int n_diag, int max_rows1, int max_rows2, size_t* bytes);

/*
 * Persistence diagrams as building blocks (torch_topological's CubicalComplex._forward on n_maps HxW maps, homology
 * dimension dim in {0, 1}), in two calls that share one workspace `ws` of tl_diagrams_workspace_bytes bytes:
 *
 * tl_diagrams_compute   the pipeline of tl_persistence_pairs (pairs of every map in gudhi's emission order, the
 *                       essential H0 class last, paired with argmax), then offsets[n_maps + 1] (int32, device) = the
 *                       exclusive scan of the per-map pair counts, and *status (int32, device, may be NULL) = the
 *                       status word (TL_STATUS_*: a NaN map or an exhausted arena; its pairs are then incomplete).
 * tl_diagrams_gather    after the host has read offsets[n_maps] and allocated P rows: map i's pairs go to rows
 *                       offsets[i] .. offsets[i+1]-1 of  pairs[P][2] = (creator, destroyer) flat pixel indices  and
 *                       diagram[P][2] = (maps[i][creator], maps[i][destroyer]), bit for bit.  `maps` and `ws` are
 *                       those of the compute call; host_offsets is the host copy of `offsets` (checked against P).
 *
 * tl_diagrams_backward  grad_maps[n_maps][H*W], fully overwritten = scatter-add of grad_diagram[P][2] into the
 *                       creator and destroyer pixels of each row (a pixel critical for several pairs adds them up).
 *
 * The [P][2] buffers (pairs, diagram, grad_diagram) are read and written as 8-byte pairs and must be 8-byte aligned.
 * Every argument error, a workspace smaller than the query asks for and a misaligned buffer included, returns TL_ERR_ARG.
 */
int tl_diagrams_workspace_bytes(int n_maps, int H, int W, int dim, size_t* bytes);
int tl_diagrams_compute(const float* maps, int n_maps, int H, int W, int dim, void* ws, size_t ws_bytes,
                        int32_t* offsets, int32_t* status, void* stream);
int tl_diagrams_gather(const float* maps, int n_maps, int H, int W, int dim, const void* ws, size_t ws_bytes,
                       const int32_t* offsets, const int32_t* host_offsets, long long P, int32_t* pairs, float* diagram,
                       void* stream);
int tl_diagrams_backward(const int32_t* pairs, const int32_t* offsets, const float* grad_diagram, long long P,
                         int n_maps, int H, int W, float* grad_maps, void* stream);

/*
 * Backward of tl_wasserstein: D1/off1, D2/off2 and match1 as tl_wasserstein took and wrote them, grad_cost[n_diag]
 * (fp32) the upstream gradient of each cost.  grad_D1[P1][2] and grad_D2[P2][2] (either may be NULL: not computed)
 * are fully overwritten with grad_cost[k] * d cost_k / d (birth, death): the gradient ot.emd2 -> pow(q) ->
 * cdist(p=inf) / distance to the diagonal give with the optimal plan.  A D1 row matched to D2 row j gets the
 * matched term and row j its negation; a row of either side matched to the diagonal gets the diagonal term.
 * D1, D2, grad_D1 and grad_D2 must be 8-byte aligned (TL_ERR_ARG otherwise).
 */
int tl_wasserstein_backward(const float* D1, const int32_t* off1, const float* D2, const int32_t* off2, int n_diag,
                            float q, const int32_t* match1, const float* grad_cost, float* grad_D1, float* grad_D2,
                            void* stream);

/*
 * Betti matching loss (Stucki et al., ICML 2023) of n_maps prediction / target pairs of HxW fp32 maps, homology
 * dimension dim in {0, 1}, sublevel filtration of the T-construction (the complex and pixel rules of tl_diagrams_*,
 * maps read as H rows of W pixels).  With C = min(pred, target): a prediction interval and a target interval are
 * matched when the intervals of the images H_dim(pred_t) -> H_dim(C_t) and H_dim(target_t) -> H_dim(C_t) born at
 * their birth cells die at the same cell of C; the two essential H0 classes (global minimum -> argmax) are always
 * matched.  Per map, in fp64, returned as fp32:
 *   cost = sum_matched (b_p - b_t)^2 + (d_p - d_t)^2 + sum_unmatched (d - b)^2 / 2.
 * Three calls share one workspace `ws` of tl_betti_workspace_bytes bytes:
 *
 * tl_betti_compute   cost[n_maps] (fp32, device), offsets[3][n_maps + 1] (int32, device) = the exclusive scans of the
 *                    per-map counts of matched, unmatched prediction and unmatched target intervals, and *status
 *                    (int32, device, may be NULL) = the status word (TL_STATUS_*: a NaN map or an exhausted arena).
 * tl_betti_gather    after the host has read the offsets (host_offsets: the same [3][n_maps + 1]; M, Kp, Kt their
 *                    totals): packed pixel indices, map i's records at rows offsets[k][i] .. offsets[k][i+1]-1 of
 *                    matched[M][4] = (pred creator, pred destroyer, target creator, target destroyer),
 *                    unmatched_pred[Kp][2] and unmatched_target[Kt][2] = (creator, destroyer).  Order within a map:
 *                    the node that owns an interval in the pixel graph (H0: birth vertex, H1: death pixel), raster
 *                    order; the H0 essential pair is the map's last matched row.
 * tl_betti_backward  grad_pred[n_maps][H*W] and, when not NULL, grad_target, fully overwritten with grad_cost[i] *
 *                    d cost_i / d map, scattered into the critical pixels of the records (atomics: a pixel critical
 *                    for several intervals adds them up).  pred / target are the maps of the compute call.
 *
 * The record buffers are read and written as 8-byte pairs and must be 8-byte aligned.  Every argument error, a
 * workspace smaller than the query asks for and a misaligned buffer included, returns TL_ERR_ARG.
 */
int tl_betti_workspace_bytes(int n_maps, int H, int W, int dim, size_t* bytes);
int tl_betti_compute(const float* pred, const float* target, int n_maps, int H, int W, int dim, void* ws, size_t ws_bytes,
                     float* cost, int32_t* offsets, int32_t* status, void* stream);
int tl_betti_gather(int n_maps, int H, int W, int dim, const void* ws, size_t ws_bytes, const int32_t* offsets,
                    const int32_t* host_offsets, long long M, long long Kp, long long Kt, int32_t* matched,
                    int32_t* unmatched_pred, int32_t* unmatched_target, void* stream);
int tl_betti_backward(const float* pred, const float* target, int n_maps, int H, int W, const int32_t* offsets,
                      const int32_t* matched, long long M, const int32_t* unmatched_pred, long long Kp,
                      const int32_t* unmatched_target, long long Kt, const float* grad_cost, float* grad_pred,
                      float* grad_target, void* stream);

/*
 * Topological prior loss (Clough et al., IPMI 2019 / TPAMI 2022) of n_maps HxW fp32 maps in homology dimension
 * dim in {0, 1}: a cost per map that asks for betti[i] features and no more, with no ground-truth map.  D is the map's
 * diagram as tl_diagrams_* computes it (same pairs, same order, the H0 essential class paired with argmax); per
 * record p = |f[destroyer] - f[creator]| (fp32 subtraction, then fabsf, values read from the map); records are
 * ranked by p descending, ties by position in D (earlier first: a stable descending sort).  In fp64, returned as fp32:
 *   cost = sum_{rank < beta} (1 - p^2) + sum_{rank >= beta} p^2 + max(0, beta - |D|)
 * (a missing interval counts as persistence 0: it adds 1 and no gradient).  The state keeps the sorted records and one
 * threshold key per map for the backward; the scratch is only live inside the forward.
 *
 * tl_prior_workspace_bytes  *state_bytes and *scratch_bytes (host pointers).
 * tl_prior_forward          betti[n_maps] (int32, device) -> cost[n_maps] (fp32, device): the persistence launch, the
 *                           sort into gudhi's emission order and one select / cost kernel.  A status bit of the
 *                           persistence launch (a NaN map, an exhausted arena) makes every cost of the call NaN; a
 *                           negative betti[i] makes cost[i] NaN.  The status word is at byte 16 of the state.
 * tl_prior_backward         grad_maps[n_maps][H*W], fully overwritten with grad_cost[i] * d cost_i / d map: for a
 *                           selected record (rank < beta) d/d death = -2 (d - b) and d/d birth = +2 (d - b), otherwise
 *                           the opposite signs, scatter-added into the critical pixels.  maps and state are those of the
 *                           forward; a map whose cost was NaN gets NaN everywhere.
 *
 * Every argument error (null pointer, a buffer smaller than the query asks for, a bad shape or dim) returns TL_ERR_ARG
 * before any launch.
 */
int tl_prior_workspace_bytes(int n_maps, int H, int W, int dim, size_t* state_bytes, size_t* scratch_bytes);
int tl_prior_forward(const float* maps, int n_maps, int H, int W, int dim, const int32_t* betti, void* state,
                     size_t state_bytes, void* scratch, size_t scratch_bytes, float* cost, void* stream);
int tl_prior_backward(const float* maps, int n_maps, int H, int W, int dim, const void* state, size_t state_bytes,
                      const float* grad_cost, float* grad_maps, void* stream);

/*
 * Exact Euclidean distance transform of n_maps HxW binary maps (H, W in [1, 4096]), unit spacing, pixel centres.
 *
 * tl_edt_workspace_bytes  *bytes (host pointer): the scratch tl_edt needs, 4 bytes per pixel.
 * tl_edt                  mask[n_maps][H][W] (uint8, device; nonzero = feature) -> out[n_maps][H][W] (fp32, device):
 *                         0 at a zero pixel; at a nonzero pixel float32(sqrt(float64(s))) with s the exact integer
 *                         squared distance to the nearest zero pixel of the same map -- what
 *                         scipy.ndimage.distance_transform_edt(m).astype(float32) gives, bit for bit, on a map with a
 *                         zero pixel.  A map without a zero pixel gets +inf everywhere.  ws must be 4-byte aligned.
 *
 * Hausdorff distance-transform loss (Karimi & Salcudean, IEEE TMI 2020) of n_maps HxW maps of fp32 logits x and
 * targets t.  Per map, p = sigmoid(x) (fp32, as torch.sigmoid), P = p > 0.5, T = t > 0.5, F(M) the distance of each
 * pixel to the nearest pixel of the other label of M if M holds both labels and 0 otherwise, D = F(P)^alpha +
 * F(T)^alpha (fp64), and
 *   cost = (1 / HW) * sum_i (p_i - t_i)^2 * D_i      (fp64, fixed order, rounded to fp32)
 *
 * tl_hausdorff_dt_workspace_bytes  *state_bytes (D, 4 bytes per pixel: written by the forward, read by the backward)
 *                                  and *scratch_bytes (8 bytes per pixel, only live inside the forward).
 * tl_hausdorff_dt_forward          cost[n_maps] (fp32, device); alpha finite and > 0.  state 4-byte, scratch 8-byte
 *                                  aligned.  A NaN logit makes its map's cost NaN.  The cost is bit-identical from
 *                                  run to run.
 * tl_hausdorff_dt_backward         grad_logits[n_maps][H][W], fully overwritten with
 *                                  grad_cost[i] * (2 / HW) * (p - t) * D * p * (1 - p); logits, target and state are
 *                                  those of the forward; state 4-byte aligned.
 *
 * Every argument error (null pointer, H or W out of range, a non-finite or non-positive alpha, a buffer smaller than
 * the query asks for or misaligned) returns TL_ERR_ARG before any launch.
 */
int tl_edt_workspace_bytes(int n_maps, int H, int W, size_t* bytes);
int tl_edt(const uint8_t* mask, int n_maps, int H, int W, void* ws, size_t ws_bytes, float* out, void* stream);
int tl_hausdorff_dt_workspace_bytes(int n_maps, int H, int W, size_t* state_bytes, size_t* scratch_bytes);
int tl_hausdorff_dt_forward(const float* logits, const float* target, int n_maps, int H, int W, double alpha,
                            void* state, size_t state_bytes, void* scratch, size_t scratch_bytes, float* cost,
                            void* stream);
int tl_hausdorff_dt_backward(const float* logits, const float* target, int n_maps, int H, int W, const void* state,
                             size_t state_bytes, const float* grad_cost, float* grad_logits, void* stream);

/*
 * Surface-distance metrics of n_maps pairs of HxW binary maps (H, W in [1, 4096]), unit spacing, pixel centres.
 * Per map: the surface S(M) = M & ~binary_erosion(M) (cross structure, outside = 0) -- the nonzero pixels with a zero
 * or an outside 4-neighbour; d_pt the exact distance sqrt(float64(s)) from each pixel of S(pred) to the nearest pixel
 * of S(target), d_tp the same the other way; n_p = |S(pred)|, n_t = |S(target)|.  Computed in fp64, rounded to fp32:
 *   hausdorff             max(max d_pt, max d_tp)
 *   hausdorff_percentile  max(pct(d_pt, q), pct(d_tp, q)), pct numpy's default (linear) percentile, q = percentile
 *   assd                  (sum d_pt + sum d_tp) / (n_p + n_t)
 *   nsd                   (#{d_pt <= tolerance} + #{d_tp <= tolerance}) / (n_p + n_t)
 * Both surfaces empty: all four NaN.  One empty: hausdorff, hausdorff_percentile and assd +inf, nsd 0.
 *
 * tl_surface_workspace_bytes  *bytes (host pointer): the scratch tl_surface_distances needs, about 16 bytes per pixel.
 * tl_surface_distances        pred, target [n_maps][H][W] (uint8, device; nonzero = foreground) -> out[4][n_maps]
 *                             (fp32, device): hausdorff, hausdorff_percentile, assd, nsd.  percentile in [0, 100],
 *                             tolerance finite and >= 0; ws 4-byte aligned.  Four launches, no host synchronisation,
 *                             bit-identical from run to run.
 *
 * Every argument error (null pointer, H or W out of range, a percentile outside [0, 100] or NaN, a negative or
 * non-finite tolerance, a workspace smaller than the query asks for or misaligned) returns TL_ERR_ARG before any launch.
 */
int tl_surface_workspace_bytes(int n_maps, int H, int W, size_t* bytes);
int tl_surface_distances(const uint8_t* pred, const uint8_t* target, int n_maps, int H, int W, double percentile,
                         double tolerance, void* ws, size_t ws_bytes, float* out, void* stream);

/*
 * Physical pixel spacing for the three entry points above (DESIGN §3.10).  spacing is a device array
 * [n_maps][2] of fp64 (sy, sx), 8-byte aligned: the size of a pixel along dim -2 (rows) and along dim -1 (columns),
 * scipy's `sampling` order.  For a zero pixel at offset (dy, dx) the squared distance is the fp64 value
 *   a = float64(dy) * sy;  b = float64(dx) * sx;  s = a*a + b*b        (each operation rounded, no contraction)
 * and the distance is float32(sqrt(min s)): what scipy.ndimage.distance_transform_edt(m, sampling=(sy, sx)) gives,
 * bit for bit.  The device cannot check the values: each must be finite and in [1e-6, 1e6], which keeps every square
 * normal in fp64 and every output finite in fp32; that is the caller's contract.
 *
 * tl_edt_spaced                    as tl_edt, with the workspace of tl_edt_workspace_bytes.
 * tl_hausdorff_dt_forward_spaced   as tl_hausdorff_dt_forward with F the spaced distance (D and the cost in physical
 *                                  units), with the buffers of tl_hausdorff_dt_workspace_bytes; the backward is
 *                                  tl_hausdorff_dt_backward.
 * tl_surface_distances_spaced      as tl_surface_distances with d_pt, d_tp the spaced distances and tolerance in the
 *                                  same units, with the workspace of tl_surface_workspace_bytes.
 *
 * Every argument error of the unspaced entry, and a null or misaligned spacing, returns TL_ERR_ARG before any launch.
 */
int tl_edt_spaced(const uint8_t* mask, int n_maps, int H, int W, const double* spacing, void* ws, size_t ws_bytes,
                  float* out, void* stream);
int tl_hausdorff_dt_forward_spaced(const float* logits, const float* target, int n_maps, int H, int W, double alpha,
                                   const double* spacing, void* state, size_t state_bytes, void* scratch,
                                   size_t scratch_bytes, float* cost, void* stream);
int tl_surface_distances_spaced(const uint8_t* pred, const uint8_t* target, int n_maps, int H, int W,
                                const double* spacing, double percentile, double tolerance, void* ws, size_t ws_bytes,
                                float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TOPOLOSS_H_ */
