// F2 (SURVEY.md 8f): the sibling loss of the reference training step,
//   seg_loss = monai.losses.DiceCELoss(sigmoid=True)          /root/reference/octsam/models/training_utils.py:32
//   train_loss = seg_loss(masks, gt_masks)                    training_utils.py:62
// as ONE read of the two [B, C, H, W] tensors per pass instead of monai's chain of elementwise kernels
// (sigmoid, three reductions, log_softmax, product, mean -- each a full round trip through HBM).
//
// monai 1.3.0 (environment.yml:224; not installed here, restated from its published source -- UNPINNED):
//   dice  = mean_{b,c} [ 1 - (2 sum_p s t + 1e-5) / (sum_p s + sum_p t + 1e-5) ],   s = sigmoid(x)
//   ce    = torch.nn.CrossEntropyLoss()(x, t) with class PROBABILITIES t over the channel axis
//         = mean_{b,p} [ - sum_c t_c (x_c - logsumexp_c' x_c') ]
//   loss  = dice + ce
// A thread owns 8 pixels of one image (strided by the block size, so every load is a coalesced 128-byte line
// per warp and channel) and walks the channels once, carrying the online-softmax state of its pixels;
// the per-channel Dice sums are reduced per warp with shuffles, per tile in shared memory and per image with
// fp64 atomics.  The backward recomputes the per-pixel log-sum-exp and writes the dense logit gradient.
// expf / logf, not the __expf / __logf intrinsics: the intrinsics' error grows with |x| (2 + 1.173 |x| ulp), and a
// trained decoder's logits reach +-20..40, where the Dice term of an empty mask is as sensitive as sum sigmoid(x) is
// small (tests/test_fused_ops_edges.py, the saturated cases).  The kernel is memory-bound either way.
#pragma once
#include "tl_common.cuh"

namespace tl {

constexpr int kDcThreads = 256;
constexpr int kDcPix = 8;           // pixels per thread
constexpr int kDcMaxC = 64;         // channels held in shared accumulators

struct DiceCeArgs {
    const float* x;        // logits  [B][C][HW]
    const float* t;        // targets [B][C][HW]
    int B, C, HW, tiles;   // tiles per image
    double* acc;           // [B][C][3] (sum s t, sum s, sum t), then [1] sum of the per-pixel CE terms
    float* loss_out;
    const float* grad_loss;
    float* gx;
};

__global__ void __launch_bounds__(kDcThreads) dice_ce_fwd_kernel(DiceCeArgs A) {
    __shared__ float s_acc[kDcMaxC][3];
    __shared__ double s_red[kDcThreads / 32];
    const int tid = threadIdx.x, lane = tid & 31;
    const int C = A.C, HW = A.HW;
    double ce_total = 0.0;
    for (int job = blockIdx.x; job < A.B * A.tiles; job += gridDim.x) {
        const int b = job / A.tiles, tile = job - b * A.tiles;
        const int p0 = tile * (kDcThreads * kDcPix) + tid;
        const float* xb = A.x + (size_t)b * C * HW;
        const float* tb = A.t + (size_t)b * C * HW;
        for (int i = tid; i < 3 * C; i += kDcThreads) (&s_acc[0][0])[i] = 0.f;
        __syncthreads();
        float m[kDcPix], s[kDcPix], dot[kDcPix], ts[kDcPix];
#pragma unroll
        for (int k = 0; k < kDcPix; ++k) { m[k] = -INFINITY; s[k] = 0.f; dot[k] = 0.f; ts[k] = 0.f; }
        for (int c = 0; c < C; ++c) {
            float xv[kDcPix], tv[kDcPix];
#pragma unroll
            for (int k = 0; k < kDcPix; ++k) {
                const int p = p0 + k * kDcThreads;
                const bool ok = p < HW;
                xv[k] = ok ? __ldg(xb + (size_t)c * HW + p) : 0.f;
                tv[k] = ok ? __ldg(tb + (size_t)c * HW + p) : 0.f;
            }
            float I = 0.f, P = 0.f, G = 0.f;
#pragma unroll
            for (int k = 0; k < kDcPix; ++k) {
                if (p0 + k * kDcThreads < HW) {
                    const float x = xv[k], t = tv[k];
                    const float sg = 1.f / (1.f + expf(-x));
                    I += sg * t; P += sg; G += t;
                    const float mn = fmaxf(m[k], x);
                    s[k] = s[k] * expf(m[k] - mn) + expf(x - mn);
                    m[k] = mn;
                    dot[k] += t * x; ts[k] += t;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                I += __shfl_down_sync(0xFFFFFFFFu, I, o); P += __shfl_down_sync(0xFFFFFFFFu, P, o); G += __shfl_down_sync(0xFFFFFFFFu, G, o);
            }
            if (lane == 0) { atomicAdd(&s_acc[c][0], I); atomicAdd(&s_acc[c][1], P); atomicAdd(&s_acc[c][2], G); }
        }
#pragma unroll
        for (int k = 0; k < kDcPix; ++k)
            if (p0 + k * kDcThreads < HW) ce_total += (double)(ts[k] * (m[k] + logf(s[k])) - dot[k]);
        __syncthreads();
        for (int i = tid; i < 3 * C; i += kDcThreads) atomicAdd(A.acc + (size_t)b * C * 3 + i, (double)(&s_acc[0][0])[i]);
        __syncthreads();
    }
    ce_total = block_sum(ce_total, s_red);
    if (tid == 0) atomicAdd(A.acc + (size_t)A.B * C * 3, ce_total);
}

__global__ void __launch_bounds__(256) dice_ce_finish_kernel(DiceCeArgs A) {
    __shared__ double s_red[8];
    double d = 0.0;
    for (int i = threadIdx.x; i < A.B * A.C; i += blockDim.x) {
        const double I = A.acc[3 * i], P = A.acc[3 * i + 1], G = A.acc[3 * i + 2];
        d += 1.0 - (2.0 * I + 1e-5) / (G + P + 1e-5);
    }
    d = block_sum(d, s_red);
    if (threadIdx.x == 0)
        *A.loss_out = (float)(d / ((double)A.B * A.C) + A.acc[(size_t)A.B * A.C * 3] / ((double)A.B * A.HW));
}

__global__ void __launch_bounds__(kDcThreads) dice_ce_bwd_kernel(DiceCeArgs A) {
    __shared__ float s_a[kDcMaxC], s_b[kDcMaxC];  // d dice_bc / d s_p = -(s_a * t_p - s_b)
    const int tid = threadIdx.x;
    const int C = A.C, HW = A.HW;
    const float g = A.grad_loss ? __ldg(A.grad_loss) : 1.f;
    const float w_dice = g / ((float)A.B * (float)C), w_ce = g / ((float)A.B * (float)HW);
    for (int job = blockIdx.x; job < A.B * A.tiles; job += gridDim.x) {
        const int b = job / A.tiles, tile = job - b * A.tiles;
        const int p0 = tile * (kDcThreads * kDcPix) + tid;
        const float* xb = A.x + (size_t)b * C * HW;
        const float* tb = A.t + (size_t)b * C * HW;
        float* gb = A.gx + (size_t)b * C * HW;
        __syncthreads();
        for (int c = tid; c < C; c += kDcThreads) {
            const double I = A.acc[((size_t)b * C + c) * 3], P = A.acc[((size_t)b * C + c) * 3 + 1], G = A.acc[((size_t)b * C + c) * 3 + 2];
            const double den = G + P + 1e-5;
            s_a[c] = (float)(2.0 / den); s_b[c] = (float)((2.0 * I + 1e-5) / (den * den));
        }
        __syncthreads();
        float m[kDcPix], s[kDcPix], ts[kDcPix];
#pragma unroll
        for (int k = 0; k < kDcPix; ++k) { m[k] = -INFINITY; s[k] = 0.f; ts[k] = 0.f; }
        for (int c = 0; c < C; ++c) {
#pragma unroll
            for (int k = 0; k < kDcPix; ++k) {
                const int p = p0 + k * kDcThreads;
                if (p < HW) {
                    const float x = __ldg(xb + (size_t)c * HW + p);
                    const float mn = fmaxf(m[k], x);
                    s[k] = s[k] * expf(m[k] - mn) + expf(x - mn);
                    m[k] = mn;
                    ts[k] += __ldg(tb + (size_t)c * HW + p);
                }
            }
        }
        for (int c = 0; c < C; ++c) {
            const float a = s_a[c], bb = s_b[c];
#pragma unroll
            for (int k = 0; k < kDcPix; ++k) {
                const int p = p0 + k * kDcThreads;
                if (p < HW) {
                    const float x = __ldg(xb + (size_t)c * HW + p), t = __ldg(tb + (size_t)c * HW + p);
                    const float sg = 1.f / (1.f + expf(-x));
                    const float soft = expf(x - m[k]) / s[k];
                    gb[(size_t)c * HW + p] = w_dice * (bb - a * t) * sg * (1.f - sg) + w_ce * (soft * ts[k] - t);
                }
            }
        }
    }
}

}  // namespace tl
