// Training loss of the hot path (forward value + both gradients):
//     L = frame_weight * (mean((c - gt)^2) + 1e-6) + w01 * mean(log v + log(1 - v)),   v = clamp(conf_coefficient, 1e-3, 1 - 1e-3)
// c = colours of the kept rays, gt looked up through the query's kept-ray list (no nonzero(), no index_select tensor).
// Reference: models/base_rendering_model.py:1114-1118 (masked MSE "+ 1e-6"), :1205-1206 (frame_weight), :1229-1240 (zero-one
// regulariser on conf_coefficient, weight 1e-4); SURVEY.md Appendix B.21.  Replaces ~30 element-wise torch launches per step.
#include "common.cuh"
#include "hnr.h"

namespace {

__global__ void __launch_bounds__(256) train_loss_kernel(const float* __restrict__ color, const float* __restrict__ gt, const int32_t* __restrict__ ray_ids,
                                                         int64_t n_rays, const float* __restrict__ confc, int64_t n_conf, float frame_weight, float w01,
                                                         double* __restrict__ partials, float* __restrict__ d_color, float* __restrict__ d_confc) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_c = n_rays * 3;
    const float kc = n_c > 0 ? frame_weight / (float)n_c : 0.f, kv = n_conf > 0 ? w01 / (float)n_conf : 0.f;
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_c; i += stride) {
        const int64_t r = i / 3;
        const int ch = (int)(i - r * 3);
        const float d = color[i] - gt[(int64_t)ray_ids[r] * 3 + ch];
        acc += (double)(kc * d * d);
        d_color[i] = 2.f * kc * d;
    }
    if (confc) {
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_conf; i += stride) {
            const float x = confc[i];
            const float v = fminf(fmaxf(x, 1e-3f), 1.f - 1e-3f);
            acc += (double)(kv * (logf(v) + logf(1.f - v)));
            // clamp passes the gradient inside [1e-3, 1 - 1e-3] (bounds included, like torch.clamp)
            d_confc[i] = (x >= 1e-3f && x <= 1.f - 1e-3f) ? kv * (1.f / v - 1.f / (1.f - v)) : 0.f;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __shared__ double red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        partials[blockIdx.x] = t;
    }
}

// one warp: the block partials summed in a fixed order (lane-strided, then a fixed shuffle tree) and rounded to fp32 once, so the loss
// does not depend on the order in which the blocks finish (fp32 atomics of the partials changed its last bit from run to run)
__global__ void train_loss_sum_kernel(const double* __restrict__ partials, int nb, float bias, float* __restrict__ loss) {
    double t = 0.0;
    for (int i = threadIdx.x; i < nb; i += 32) t += partials[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) *loss = (float)(t + (double)bias);
}

}  // namespace

// loss (1 float) = the training loss; d_color (n_rays,3) and d_confc (n_conf) receive dL/dcolor, dL/dconf_coefficient.
// gt: (R,3) colours of ALL rays, ray_ids: (n_rays) int32 kept-ray list.  confc may be NULL (no regulariser).
// partials: scratch of HNR_TRAIN_LOSS_PARTIALS doubles (one per block of the first launch).
extern "C" int hnr_train_loss(const float* color, const float* gt, const int32_t* ray_ids, int64_t n_rays, const float* confc, int64_t n_conf,
                              float frame_weight, float zero_one_weight, float* loss, double* partials, float* d_color, float* d_confc,
                              void* stream) {
    HNR_CHECK_ARG(n_rays >= 0 && n_conf >= 0, "train_loss: bad sizes");
    int64_t work = n_rays * 3 > n_conf ? n_rays * 3 : n_conf;
    int64_t nb = hnr_cdiv(work, 256 * 4);
    if (nb < 1) nb = 1;
    if (nb > 2 * HNR_NUM_SMS) nb = 2 * HNR_NUM_SMS;
    static_assert(2 * HNR_NUM_SMS <= HNR_TRAIN_LOSS_PARTIALS, "train_loss: partials scratch too small");
    train_loss_kernel<<<(unsigned)nb, 256, 0, (cudaStream_t)stream>>>(color, gt, ray_ids, n_rays, confc, confc ? n_conf : 0, frame_weight,
                                                                    zero_one_weight, partials, d_color, d_confc);
    train_loss_sum_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(partials, (int)nb, n_rays > 0 ? frame_weight * 1e-6f : 0.f, loss);
    HNR_CHECK_LAUNCH("train_loss");
    return HNR_OK;
}
