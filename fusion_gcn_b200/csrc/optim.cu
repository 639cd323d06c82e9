// Multi-tensor optimizer steps (SURVEY 8 f4): ONE launch updates every parameter tensor of a group.
//
// The reference builds torch.optim.{SGD, Adam, AdamW} over model.parameters() (torch_src/session_helper.py:48-82) and steps them
// after every batch (torch_src/session/procedures/step.py:48-49), under GradScaler when --mixed_precision is set (:67-71).  The
// AGCN model has 274 parameter tensors, most of them a few hundred floats: per-tensor kernels leave hundreds of launches of a few
// microseconds behind the 60 ms step.  Here the tensors stay where PyTorch put them (state-dict / checkpoint layout untouched); a
// device table of (param, grad, state1, state2, numel) rows and a list of (tensor, chunk) work items let one grid walk all of them.
// GradScaler: torch hands optimizers that declare _step_supports_amp_scaling the device scalars `grad_scale` and `found_inf`; the
// unscale (g / scale) and the skip-on-overflow are done here, so no host synchronisation is needed and the step is graph-capturable.
// Arithmetic follows torch/optim/sgd.py (_single_tensor_sgd), torch/optim/adam.py (_single_tensor_adam, capturable form) and
// torch/optim/asgd.py (_single_tensor_asgd, capturable form).  `maximize` negates the unscaled gradient, as torch does before weight
// decay: it is folded into the unscale factor, (-s) * g == -(s * g) exactly.
#include "common.cuh"

namespace agcn {

constexpr int kOptChunk = 4096;          // elements per work item
constexpr int kOptThreads = 256;

struct OptRow { float* p; const float* g; float* s1; float* s2; long long n; };
// AMSGrad keeps a third state tensor (max_exp_avg_sq); only its Adam table carries the extra column
struct AmsgradRow { float* p; const float* g; float* s1; float* s2; float* s3; long long n; };

// hyper-parameters arrive as doubles (Python floats) and are rounded to fp32 only where torch rounds them: 1 - beta and the bias
// corrections are formed in double first (1.f - 0.999f is 1.3e-5 away from float(1 - 0.999))
struct SgdHyper { double lr, momentum, dampening, weight_decay; int nesterov, first, maximize; };
struct AdamHyper { double lr, beta1, beta2, eps, weight_decay; int decoupled, maximize; };
struct AsgdHyper { double lr, lambd, alpha, t0, weight_decay; int maximize; };

template <typename Row, typename F>
__device__ __forceinline__ void for_chunk(const Row& t, long long base, F f) {
    const long long end = (base + kOptChunk < t.n) ? base + kOptChunk : t.n;
    for (long long i = base + threadIdx.x; i < end; i += kOptThreads) f(i);
}

__global__ void __launch_bounds__(kOptThreads)
sgd_kernel(const OptRow* __restrict__ table, const int2* __restrict__ items, SgdHyper h, const float* __restrict__ lr_dev,
           const float* __restrict__ grad_scale, const float* __restrict__ found_inf) {
    if (found_inf != nullptr && *found_inf != 0.f) return;          // GradScaler: skip the whole step on overflow
    const int2 it = items[blockIdx.x];
    const OptRow t = table[it.x];
    const float lr = lr_dev != nullptr ? *lr_dev : (float)h.lr;
    float inv_scale = grad_scale != nullptr ? 1.f / *grad_scale : 1.f;
    if (h.maximize) inv_scale = -inv_scale;
    const float wd = (float)h.weight_decay, mom = (float)h.momentum, damp1 = (float)(1.0 - h.dampening);
    for_chunk(t, (long long)it.y * kOptChunk, [&](long long i) {
        const float p = t.p[i];
        float g = t.g[i] * inv_scale;
        if (wd != 0.f) g = fmaf(wd, p, g);
        if (mom != 0.f) {
            float buf = h.first ? g : fmaf(mom, t.s1[i], damp1 * g);
            t.s1[i] = buf;
            g = h.nesterov ? fmaf(mom, buf, g) : buf;
        }
        t.p[i] = fmaf(-lr, g, p);
    });
}

template <bool kAmsgrad> struct AdamRowOf { using type = OptRow; };
template <> struct AdamRowOf<true> { using type = AmsgradRow; };

template <bool kAmsgrad>
__global__ void __launch_bounds__(kOptThreads)
adam_kernel(const typename AdamRowOf<kAmsgrad>::type* __restrict__ table, const int2* __restrict__ items, AdamHyper h,
            const float* __restrict__ lr_dev, const float* __restrict__ step_dev, const float* __restrict__ grad_scale,
            const float* __restrict__ found_inf) {
    if (found_inf != nullptr && *found_inf != 0.f) return;
    const int2 it = items[blockIdx.x];
    const auto t = table[it.x];
    const double lr_d = lr_dev != nullptr ? (double)*lr_dev : h.lr;
    float inv_scale = grad_scale != nullptr ? 1.f / *grad_scale : 1.f;
    if (h.maximize) inv_scale = -inv_scale;
    const double step = (double)*step_dev + 1.0;                     // steps completed so far + this one
    const float step_size = (float)(lr_d / (1.0 - pow(h.beta1, step)));
    const float bc2_sqrt = (float)sqrt(1.0 - pow(h.beta2, step));
    const float b1 = (float)h.beta1, b2 = (float)h.beta2, omb1 = (float)(1.0 - h.beta1), omb2 = (float)(1.0 - h.beta2);
    const float wd = (float)h.weight_decay, eps = (float)h.eps, decay = (float)(1.0 - lr_d * h.weight_decay);
    for_chunk(t, (long long)it.y * kOptChunk, [&](long long i) {
        float p = t.p[i];
        float g = t.g[i] * inv_scale;
        if (h.decoupled) p *= decay;                                 // AdamW
        else if (wd != 0.f) g = fmaf(wd, p, g);
        const float m0 = t.s1[i];
        const float m = fmaf(omb1, g - m0, m0);                      // exp_avg.lerp_(grad, 1 - beta1)
        const float v = fmaf(omb2 * g, g, b2 * t.s2[i]);             // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
        t.s1[i] = m;
        t.s2[i] = v;
        float vmax = v;
        if constexpr (kAmsgrad) {                                    // max_exp_avg_sq = maximum(max_exp_avg_sq, exp_avg_sq)
            const float v0 = t.s3[i];
            vmax = (v >= v0 || v != v) ? v : v0;                     // NaN from either side propagates, as torch.maximum
            t.s3[i] = vmax;
        }
        const float denom = sqrtf(vmax) / bc2_sqrt + eps;
        t.p[i] = fmaf(-step_size, m / denom, p);
    });
    (void)b1;
}

// ASGD, rows { param, grad, ax, -, numel }.  eta / mu / step are ONE set of device scalars shared by the group; every block reads
// eta and mu, and the last block to finish (counted on *done, which it resets to zero) advances them once:
//   step += 1;  eta = lr / (1 + lambd * lr * step)^alpha;  mu = 1 / max(1, step - t0)
// so one launch is the whole step, with nothing for the host to do afterwards (GradScaler's skip included).
__global__ void __launch_bounds__(kOptThreads)
asgd_kernel(const OptRow* __restrict__ table, const int2* __restrict__ items, AsgdHyper h, const float* __restrict__ lr_dev,
            float* eta_dev, float* mu_dev, float* step_dev, int* done, const float* __restrict__ grad_scale,
            const float* __restrict__ found_inf) {
    if (found_inf != nullptr && *found_inf != 0.f) return;          // skipped: parameters, ax and the scalars all stay
    const int2 it = items[blockIdx.x];
    const OptRow t = table[it.x];
    float inv_scale = grad_scale != nullptr ? 1.f / *grad_scale : 1.f;
    if (h.maximize) inv_scale = -inv_scale;
    const float eta = *eta_dev, mu = *mu_dev;
    const float wd = (float)h.weight_decay;
    const float decay = 1.f - (float)h.lambd * eta;                 // param.mul_(1 - lambd * eta) on the fp32 eta tensor
    for_chunk(t, (long long)it.y * kOptChunk, [&](long long i) {
        float g = t.g[i] * inv_scale;
        float p = t.p[i];
        if (wd != 0.f) g = fmaf(wd, p, g);
        p = fmaf(-eta, g, p * decay);                                // param.addcmul_(grad, eta, value=-1)
        t.p[i] = p;
        const float ax = t.s1[i];
        t.s1[i] = fmaf(p - ax, mu, ax);                              // ax.add_(param.sub(ax).mul_(mu))
    });
    __syncthreads();                                                 // every thread of this block has used eta and mu
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(done, 1) == (int)gridDim.x - 1) {              // all other blocks are past their reads of eta / mu
            const double lr = lr_dev != nullptr ? (double)*lr_dev : h.lr;
            const float step = *step_dev + 1.f;
            *step_dev = step;
            *eta_dev = (float)(lr / pow(1.0 + h.lambd * lr * (double)step, h.alpha));
            *mu_dev = (float)(1.0 / fmax(1.0, (double)step - h.t0));
            *done = 0;
        }
    }
}

// flat[off ...] <-> tensor copies for the gradient buckets of the data-parallel all-reduce: rows { flat slice, tensor, -, -, numel }
// (OptRow with p = flat slice, g = tensor).  to_flat: flat = tensor;  else: tensor = flat * scale (the 1 / world averaging).
__global__ void __launch_bounds__(kOptThreads)
bucket_copy_kernel(const OptRow* __restrict__ table, const int2* __restrict__ items, int to_flat, float scale) {
    const int2 it = items[blockIdx.x];
    const OptRow t = table[it.x];
    float* tensor = const_cast<float*>(t.g);
    for_chunk(t, (long long)it.y * kOptChunk, [&](long long i) {
        if (to_flat) t.p[i] = tensor[i];
        else tensor[i] = t.p[i] * scale;
    });
}

static int check_table(const void* table, const int* items, int nitems, const char* what) {
    AGCN_REQUIRE(table && items, AGCN_ERR_NULL, "%s: null table / work list", what);
    AGCN_REQUIRE(nitems > 0, AGCN_ERR_BAD_SHAPE, "%s: empty work list", what);
    AGCN_REQUIRE((reinterpret_cast<uintptr_t>(table) & 7u) == 0 && (reinterpret_cast<uintptr_t>(items) & 7u) == 0, AGCN_ERR_MISALIGNED,
                 "%s: table / work list not 8-byte aligned", what);
    return AGCN_OK;
}

}  // namespace agcn

using namespace agcn;

extern "C" AGCN_API int agcn_optim_chunk(void) { return kOptChunk; }

extern "C" AGCN_API int agcn_optim_sgd(const void* table, const int* items, int nitems, double lr, const float* lr_dev,
                                       double momentum, double dampening, double weight_decay, int nesterov, int first_step, int maximize,
                                       const float* grad_scale, const float* found_inf, void* stream) {
    int rc = check_table(table, items, nitems, "agcn_optim_sgd");
    if (rc) return rc;
    AGCN_REQUIRE(!nesterov || (momentum > 0.0 && dampening == 0.0), AGCN_ERR_UNSUPPORTED,
                 "agcn_optim_sgd: Nesterov momentum requires a momentum and zero dampening");       // torch/optim/sgd.py raises the same
    SgdHyper h{lr, momentum, dampening, weight_decay, nesterov, first_step, maximize};
    sgd_kernel<<<nitems, kOptThreads, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const OptRow*>(table), reinterpret_cast<const int2*>(items),
                                                                              h, lr_dev, grad_scale, found_inf);
    return check_launch("agcn_optim_sgd");
}

extern "C" AGCN_API int agcn_optim_adam(const void* table, const int* items, int nitems, double lr, const float* lr_dev,
                                        double beta1, double beta2, double eps, double weight_decay, int decoupled, int amsgrad,
                                        int maximize, const float* step_dev, const float* grad_scale, const float* found_inf,
                                        void* stream) {
    int rc = check_table(table, items, nitems, "agcn_optim_adam");
    if (rc) return rc;
    AGCN_REQUIRE(step_dev != nullptr, AGCN_ERR_NULL, "agcn_optim_adam: null step counter");
    AdamHyper h{lr, beta1, beta2, eps, weight_decay, decoupled, maximize};
    const int2* work = reinterpret_cast<const int2*>(items);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (amsgrad)
        adam_kernel<true><<<nitems, kOptThreads, 0, s>>>(static_cast<const AmsgradRow*>(table), work, h, lr_dev, step_dev, grad_scale, found_inf);
    else
        adam_kernel<false><<<nitems, kOptThreads, 0, s>>>(static_cast<const OptRow*>(table), work, h, lr_dev, step_dev, grad_scale, found_inf);
    return check_launch("agcn_optim_adam");
}

extern "C" AGCN_API int agcn_optim_asgd(const void* table, const int* items, int nitems, double lr, const float* lr_dev,
                                        double lambd, double alpha, double t0, double weight_decay, int maximize,
                                        float* eta, float* mu, float* step, int* done, const float* grad_scale, const float* found_inf,
                                        void* stream) {
    int rc = check_table(table, items, nitems, "agcn_optim_asgd");
    if (rc) return rc;
    AGCN_REQUIRE(eta && mu && step && done, AGCN_ERR_NULL, "agcn_optim_asgd: null eta / mu / step / done scalar");
    AsgdHyper h{lr, lambd, alpha, t0, weight_decay, maximize};
    asgd_kernel<<<nitems, kOptThreads, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const OptRow*>(table), reinterpret_cast<const int2*>(items),
                                                                               h, lr_dev, eta, mu, step, done, grad_scale, found_inf);
    return check_launch("agcn_optim_asgd");
}

extern "C" AGCN_API int agcn_bucket_copy(const void* table, const int* items, int nitems, int to_flat, float scale, void* stream) {
    int rc = check_table(table, items, nitems, "agcn_bucket_copy");
    if (rc) return rc;
    bucket_copy_kernel<<<nitems, kOptThreads, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const OptRow*>(table), reinterpret_cast<const int2*>(items),
                                                                                 to_flat, scale);
    return check_launch("agcn_bucket_copy");
}
