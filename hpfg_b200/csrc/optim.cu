// Flat-buffer optimiser passes: EMA teacher update (utils/utils.py:82-86), torch.optim.SGD momentum step
// (utils/__init__.py:14-16) and the two fused, torch.optim.Adam / AdamW (utils/__init__.py:13-49) with an optional
// fused EMA.  Pure HBM streaming kernels: 128-bit loads/stores, grid sized as a multiple of the SM count, grid-stride
// loop.  Algorithmic traffic: EMA 12 B/param, SGD 20 B/param (first step 16), fused 28 B/param; Adam 28 B/param,
// Adam + EMA 36 B/param.
#include "common.cuh"

namespace hpfg {

__device__ __forceinline__ float4 ldg4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }

// ema <- alpha*ema + (1-alpha)*p, rounded the way `ema.mul_(alpha).add_(p, alpha=1-alpha)` rounds:
// the product alpha*ema is rounded to fp32 first, then (1-alpha)*p is added.
__device__ __forceinline__ float ema1(float e, float p, float alpha, float one_minus) {
    return __fmaf_rn(one_minus, p, __fmul_rn(alpha, e));
}

__global__ void __launch_bounds__(256) ema_kernel(float *__restrict__ ema, const float *__restrict__ param,
                                                  int64_t n, float alpha, float one_minus) {
    pdl_prologue();
    const int64_t n4 = n >> 2;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 e = *reinterpret_cast<float4 *>(ema + 4 * i);
        const float4 p = ldg4(param + 4 * i);
        e.x = ema1(e.x, p.x, alpha, one_minus);
        e.y = ema1(e.y, p.y, alpha, one_minus);
        e.z = ema1(e.z, p.z, alpha, one_minus);
        e.w = ema1(e.w, p.w, alpha, one_minus);
        *reinterpret_cast<float4 *>(ema + 4 * i) = e;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const int64_t i = (n4 << 2) + threadIdx.x;
        ema[i] = ema1(ema[i], param[i], alpha, one_minus);
    }
}

// torch.optim.SGD (foreach, momentum, weight_decay; no nesterov, dampening 0):
//   d = g*scale + wd*p ; buf = first ? d : mom*buf + d ; p = p - lr*buf
struct SgdArgs {
    float lr, momentum, weight_decay, grad_scale, ema_alpha, ema_one_minus;
    int first_step;
    const float *dyn;      // optional device block {lr, ema_alpha, 1 - ema_alpha}: overrides the by-value fields (CUDA-graph replays)
};

template <bool kEma>
__device__ __forceinline__ void sgd1(float &p, float g, float &buf, float &e, const SgdArgs &a) {
    float d = __fmaf_rn(a.weight_decay, p, g * a.grad_scale);
    buf = a.first_step ? d : __fmaf_rn(a.momentum, buf, d);
    p = __fmaf_rn(-a.lr, buf, p);
    if (kEma) e = ema1(e, p, a.ema_alpha, a.ema_one_minus);
}

template <bool kEma>
__global__ void __launch_bounds__(256) sgd_kernel(float *__restrict__ param, const float *__restrict__ grad,
                                                  float *__restrict__ buf, float *__restrict__ ema, int64_t n,
                                                  SgdArgs a) {
    pdl_prologue();
    if (a.dyn) {
        a.lr = a.dyn[0];
        if (kEma) { a.ema_alpha = a.dyn[1]; a.ema_one_minus = a.dyn[2]; }
    }
    const int64_t n4 = n >> 2;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 p = *reinterpret_cast<float4 *>(param + 4 * i);
        const float4 g = ldg4(grad + 4 * i);
        float4 b = a.first_step ? make_float4(0, 0, 0, 0) : *reinterpret_cast<float4 *>(buf + 4 * i);
        float4 e = make_float4(0, 0, 0, 0);
        if (kEma) e = *reinterpret_cast<float4 *>(ema + 4 * i);
        sgd1<kEma>(p.x, g.x, b.x, e.x, a);
        sgd1<kEma>(p.y, g.y, b.y, e.y, a);
        sgd1<kEma>(p.z, g.z, b.z, e.z, a);
        sgd1<kEma>(p.w, g.w, b.w, e.w, a);
        *reinterpret_cast<float4 *>(param + 4 * i) = p;
        *reinterpret_cast<float4 *>(buf + 4 * i) = b;
        if (kEma) *reinterpret_cast<float4 *>(ema + 4 * i) = e;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const int64_t i = (n4 << 2) + threadIdx.x;
        float e = kEma ? ema[i] : 0.f, b = a.first_step ? 0.f : buf[i], p = param[i];
        sgd1<kEma>(p, grad[i], b, e, a);
        param[i] = p;
        buf[i] = b;
        if (kEma) ema[i] = e;
    }
}

// torch.optim.Adam / AdamW (foreach, non-capturable, no amsgrad / maximize), per element in the order of
// torch/optim/adam.py:_multi_tensor_adam:
//   g = grad*scale ; Adam: g = g + wd*p | AdamW: p = p*(1 - lr*wd)
//   m = lerp(m, g, 1 - beta1) ; v = v*beta2 ; v = v + (1 - beta2)*(g*g)
//   p = p + step_size*(m / (sqrt(v)/bc2_sqrt + eps))      step_size = -lr/(1 - beta1^t), bc2_sqrt = sqrt(1 - beta2^t)
// addcmul_ / addcdiv_ are explicit fmas in ATen (DeviceAddCmulCdiv.cuh); lerp (ATen Lerp.h) and the L2 add are
// contracted to fmas by nvcc in torch's build (profiles/adam_microbench.txt).  The 1 - beta complements and the
// step-dependent scalars are computed in double on the host, as torch computes them in Python.
struct AdamArgs {
    float one_minus_beta1, beta2, one_minus_beta2, eps, weight_decay, grad_scale;
    float step_size, bc2_sqrt, decay_factor, ema_alpha, ema_one_minus;
    int decoupled;
    const float *dyn;      // optional device block {step_size, bc2_sqrt, decay_factor, ema_alpha, 1 - ema_alpha} (CUDA-graph replays)
};

template <bool kEma>
__device__ __forceinline__ void adam1(float &p, float g, float &m, float &v, float &e, const AdamArgs &a) {
    g = __fmul_rn(g, a.grad_scale);
    if (a.weight_decay != 0.f) {
        if (a.decoupled) p = __fmul_rn(p, a.decay_factor);
        else g = __fmaf_rn(a.weight_decay, p, g);
    }
    const float w = a.one_minus_beta1;
    m = w < 0.5f ? __fmaf_rn(w, __fsub_rn(g, m), m) : __fmaf_rn(-__fsub_rn(g, m), __fsub_rn(1.f, w), g);
    v = __fmaf_rn(a.one_minus_beta2, __fmul_rn(g, g), __fmul_rn(v, a.beta2));
    const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), a.bc2_sqrt), a.eps);
    p = __fmaf_rn(a.step_size, __fdiv_rn(m, denom), p);
    if (kEma) e = ema1(e, p, a.ema_alpha, a.ema_one_minus);
}

template <bool kEma>
__global__ void __launch_bounds__(256) adam_kernel(float *__restrict__ param, const float *__restrict__ grad,
                                                   float *__restrict__ exp_avg, float *__restrict__ exp_avg_sq,
                                                   float *__restrict__ ema, int64_t n, AdamArgs a) {
    pdl_prologue();
    if (a.dyn) {
        a.step_size = a.dyn[0];
        a.bc2_sqrt = a.dyn[1];
        a.decay_factor = a.dyn[2];
        if (kEma) { a.ema_alpha = a.dyn[3]; a.ema_one_minus = a.dyn[4]; }
    }
    const int64_t n4 = n >> 2;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 p = *reinterpret_cast<float4 *>(param + 4 * i);
        const float4 g = ldg4(grad + 4 * i);
        float4 m = *reinterpret_cast<float4 *>(exp_avg + 4 * i);
        float4 v = *reinterpret_cast<float4 *>(exp_avg_sq + 4 * i);
        float4 e = make_float4(0, 0, 0, 0);
        if (kEma) e = *reinterpret_cast<float4 *>(ema + 4 * i);
        adam1<kEma>(p.x, g.x, m.x, v.x, e.x, a);
        adam1<kEma>(p.y, g.y, m.y, v.y, e.y, a);
        adam1<kEma>(p.z, g.z, m.z, v.z, e.z, a);
        adam1<kEma>(p.w, g.w, m.w, v.w, e.w, a);
        *reinterpret_cast<float4 *>(param + 4 * i) = p;
        *reinterpret_cast<float4 *>(exp_avg + 4 * i) = m;
        *reinterpret_cast<float4 *>(exp_avg_sq + 4 * i) = v;
        if (kEma) *reinterpret_cast<float4 *>(ema + 4 * i) = e;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const int64_t i = (n4 << 2) + threadIdx.x;
        float e = kEma ? ema[i] : 0.f, p = param[i], m = exp_avg[i], v = exp_avg_sq[i];
        adam1<kEma>(p, grad[i], m, v, e, a);
        param[i] = p;
        exp_avg[i] = m;
        exp_avg_sq[i] = v;
        if (kEma) ema[i] = e;
    }
}

static int flat_grid(int64_t n) {
    int64_t blocks = (n / 4 + 255) / 256;
    int64_t cap = (int64_t)kNumSMs * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace hpfg

using namespace hpfg;

extern "C" int hpfg_ema_update(float *ema, const float *param, int64_t n, float alpha, void *stream) {
    HPFG_REQUIRE(ema && param && n >= 0, "hpfg_ema_update: null buffer");
    HPFG_REQUIRE(aligned16(ema) && aligned16(param), "hpfg_ema_update: buffers must be 16-byte aligned");
    if (n == 0) return HPFG_OK;
    ProfScope _prof(PROF_OPTIM, (cudaStream_t)stream);
    HPFG_CUDA_CHECK(launch_pdl(ema_kernel, flat_grid(n), 256, 0, (cudaStream_t)stream, ema, param, n, alpha, 1.0f - alpha));
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}

static int sgd_launch(const char *what, float *param, const float *grad, float *momentum_buf, float *ema, int64_t n,
                      const SgdArgs &a, void *stream) {
    HPFG_REQUIRE(param && grad && momentum_buf && n >= 0, std::string(what) + ": null buffer");
    HPFG_REQUIRE(aligned16(param) && aligned16(grad) && aligned16(momentum_buf) && (!ema || aligned16(ema)),
                 std::string(what) + ": buffers must be 16-byte aligned");
    if (n == 0) return HPFG_OK;
    ProfScope _prof(PROF_OPTIM, (cudaStream_t)stream);
    if (ema)
        HPFG_CUDA_CHECK(launch_pdl(sgd_kernel<true>, flat_grid(n), 256, 0, (cudaStream_t)stream, param, grad, momentum_buf, ema, n, a));
    else
        HPFG_CUDA_CHECK(launch_pdl(sgd_kernel<false>, flat_grid(n), 256, 0, (cudaStream_t)stream, param, grad, momentum_buf, (float *)nullptr, n, a));
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}

extern "C" int hpfg_sgd_momentum(float *param, const float *grad, float *momentum_buf, int64_t n, float lr,
                                 float momentum, float weight_decay, float grad_scale, int first_step,
                                 void *stream) {
    SgdArgs a{lr, momentum, weight_decay, grad_scale, 0.f, 0.f, first_step, nullptr};
    return sgd_launch("hpfg_sgd_momentum", param, grad, momentum_buf, nullptr, n, a, stream);
}

extern "C" int hpfg_sgd_momentum_ema(float *param, const float *grad, float *momentum_buf, float *ema, int64_t n,
                                     float lr, float momentum, float weight_decay, float grad_scale,
                                     int first_step, float ema_alpha, void *stream) {
    HPFG_REQUIRE(ema, "hpfg_sgd_momentum_ema: null buffer");
    SgdArgs a{lr, momentum, weight_decay, grad_scale, ema_alpha, 1.0f - ema_alpha, first_step, nullptr};
    return sgd_launch("hpfg_sgd_momentum_ema", param, grad, momentum_buf, ema, n, a, stream);
}

extern "C" int hpfg_sgd_momentum_ema_dv(float *param, const float *grad, float *momentum_buf, float *ema, int64_t n,
                                        float momentum, float weight_decay, float grad_scale, int first_step,
                                        const float *lr_alpha_dev, void *stream) {
    HPFG_REQUIRE(ema && lr_alpha_dev, "hpfg_sgd_momentum_ema_dv: null buffer");
    SgdArgs a{0.f, momentum, weight_decay, grad_scale, 0.f, 0.f, first_step, lr_alpha_dev};
    return sgd_launch("hpfg_sgd_momentum_ema_dv", param, grad, momentum_buf, ema, n, a, stream);
}

extern "C" int hpfg_sgd_momentum_dv(float *param, const float *grad, float *momentum_buf, int64_t n, float momentum,
                                    float weight_decay, float grad_scale, int first_step, const float *lr_dev,
                                    void *stream) {
    HPFG_REQUIRE(lr_dev, "hpfg_sgd_momentum_dv: null buffer");
    SgdArgs a{0.f, momentum, weight_decay, grad_scale, 0.f, 0.f, first_step, lr_dev};
    return sgd_launch("hpfg_sgd_momentum_dv", param, grad, momentum_buf, nullptr, n, a, stream);
}

static int adam_launch(const char *what, float *param, const float *grad, float *exp_avg, float *exp_avg_sq, float *ema,
                       int64_t n, const AdamArgs &a, void *stream) {
    HPFG_REQUIRE(param && grad && exp_avg && exp_avg_sq && n >= 0, std::string(what) + ": null buffer");
    HPFG_REQUIRE(aligned16(param) && aligned16(grad) && aligned16(exp_avg) && aligned16(exp_avg_sq) && (!ema || aligned16(ema)),
                 std::string(what) + ": buffers must be 16-byte aligned");
    if (n == 0) return HPFG_OK;
    ProfScope _prof(PROF_OPTIM, (cudaStream_t)stream);
    if (ema)
        HPFG_CUDA_CHECK(launch_pdl(adam_kernel<true>, flat_grid(n), 256, 0, (cudaStream_t)stream, param, grad, exp_avg, exp_avg_sq, ema, n, a));
    else
        HPFG_CUDA_CHECK(launch_pdl(adam_kernel<false>, flat_grid(n), 256, 0, (cudaStream_t)stream, param, grad, exp_avg, exp_avg_sq, (float *)nullptr, n, a));
    HPFG_LAUNCH_CHECK();
    return HPFG_OK;
}

extern "C" int hpfg_adam(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, float *ema, int64_t n,
                         float one_minus_beta1, float beta2, float one_minus_beta2, float eps, float weight_decay,
                         int decoupled, float grad_scale, float step_size, float bc2_sqrt, float decay_factor,
                         float ema_alpha, void *stream) {
    AdamArgs a{one_minus_beta1, beta2, one_minus_beta2, eps, weight_decay, grad_scale, step_size, bc2_sqrt, decay_factor,
               ema_alpha, 1.0f - ema_alpha, decoupled, nullptr};
    return adam_launch("hpfg_adam", param, grad, exp_avg, exp_avg_sq, ema, n, a, stream);
}

extern "C" int hpfg_adam_dv(float *param, const float *grad, float *exp_avg, float *exp_avg_sq, float *ema, int64_t n,
                            float one_minus_beta1, float beta2, float one_minus_beta2, float eps, float weight_decay,
                            int decoupled, float grad_scale, const float *dyn, void *stream) {
    HPFG_REQUIRE(dyn, "hpfg_adam_dv: null buffer");
    AdamArgs a{one_minus_beta1, beta2, one_minus_beta2, eps, weight_decay, grad_scale, 0.f, 0.f, 0.f, 0.f, 0.f, decoupled, dyn};
    return adam_launch("hpfg_adam_dv", param, grad, exp_avg, exp_avg_sq, ema, n, a, stream);
}
