// F3: the optimiser step of the trainer (torch.optim.Adam(lr=5e-4, betas=(0.9,0.999)), run_nerf_uncertainty_NF.py:339,
// 1065-1077) as ONE launch over all parameter tensors, with the data-parallel 1/world gradient scaling folded in.
#include "common.cuh"

namespace cfn {

constexpr int kAdamMaxTensors = 64;
struct AdamTable {
  float* p[kAdamMaxTensors];
  const float* g[kAdamMaxTensors];
  float* m[kAdamMaxTensors];
  float* v[kAdamMaxTensors];
  int64_t n[kAdamMaxTensors];
};

// The learning rate and bias corrections come from the device clock `state` (see adam_advance_kernel) when it is given,
// else from the host values lr, bc1 = 1 - beta1^step and bc2_sqrt = sqrt(1 - beta2^step).  The launch bounds keep it at 32
// registers, i.e. full occupancy for this bandwidth-bound loop (the two-way prologue alone would take 34).
__global__ void __launch_bounds__(256, 8) adam_kernel(AdamTable t, const float* __restrict__ state, float lr, float bc1, float bc2_sqrt, float beta1,
                            float beta2, float eps, float grad_scale) {
  const int ti = blockIdx.y;
  const int64_t n = t.n[ti];
  float* __restrict__ p = t.p[ti];
  const float* __restrict__ g = t.g[ti];
  float* __restrict__ m = t.m[ti];
  float* __restrict__ v = t.v[ti];
  const float step_size = state ? state[1] / state[2] : lr / bc1;
  const float bc2 = state ? state[3] : bc2_sqrt;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i] * grad_scale;
    const float mi = m[i] + (gi - m[i]) * (1.0f - beta1);          // exp_avg.lerp_(grad, 1 - beta1)
    const float vi = v[i] * beta2 + (1.0f - beta2) * gi * gi;      // exp_avg_sq.mul_(beta2).addcmul_(g, g, 1 - beta2)
    const float denom = sqrtf(vi) / bc2 + eps;
    m[i] = mi;
    v[i] = vi;
    p[i] = p[i] - step_size * (mi / denom);
  }
}

// ---- device-resident optimiser clock: the same step inside a CUDA graph -----------------------------------------
// state (device, 4 floats) = [step count, learning rate of this step, 1 - beta1^step, sqrt(1 - beta2^step)].  One thread
// advances it; the update kernel reads it, so neither the step count nor the decayed learning rate is baked into a
// captured launch.  lr(t) = lr0 * decay_rate^(max(t - 2, 0) / decay_steps): the reference applies the schedule AFTER
// optimizer.step() with a global_step that lags the iteration by one (run_nerf_uncertainty_NF.py:931, 1073-1077, 1198).
__global__ void adam_advance_kernel(float* __restrict__ state, float lr0, float decay_rate, float decay_steps, float beta1,
                                    float beta2) {
  const float t = state[0] + 1.0f;
  state[0] = t;
  state[1] = (decay_steps > 0.f) ? lr0 * powf(decay_rate, fmaxf(t - 2.0f, 0.f) / decay_steps) : lr0;
  state[2] = 1.0f - powf(beta1, t);
  state[3] = sqrtf(1.0f - powf(beta2, t));
}

// adam_kernel over every tensor, at most kAdamMaxTensors per launch
static int adam_update(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                       float* const* exp_avg_sq, const int64_t* numels, const float* state, float lr, float bc1,
                       float bc2_sqrt, float beta1, float beta2, float eps, float grad_scale, cudaStream_t s) {
  for (int base = 0; base < n_tensors; base += kAdamMaxTensors) {
    AdamTable t;
    const int cnt = n_tensors - base < kAdamMaxTensors ? n_tensors - base : kAdamMaxTensors;
    int64_t biggest = 0;
    for (int i = 0; i < cnt; ++i) {
      CFN_CHECK_ARG(params[base + i] && grads[base + i] && exp_avg[base + i] && exp_avg_sq[base + i], "adam: null tensor %d",
                    base + i);
      t.p[i] = params[base + i]; t.g[i] = grads[base + i]; t.m[i] = exp_avg[base + i]; t.v[i] = exp_avg_sq[base + i];
      t.n[i] = numels[base + i];
      if (t.n[i] > biggest) biggest = t.n[i];
    }
    if (cnt == 0 || biggest == 0) continue;
    int64_t bx = (biggest + 1023) / 1024;
    if (bx > 148 * 4) bx = 148 * 4;
    adam_kernel<<<dim3((unsigned)bx, (unsigned)cnt), 256, 0, s>>>(t, state, lr, bc1, bc2_sqrt, beta1, beta2, eps,
                                                                   grad_scale);
    CFN_LAUNCH_CHECK();
  }
  return CFN_OK;
}

int launch_adam_dev(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                    float* const* exp_avg_sq, const int64_t* numels, float* state, float lr0, float decay_rate,
                    float decay_steps, float beta1, float beta2, float eps, float grad_scale, cudaStream_t s) {
  CFN_CHECK_ARG(n_tensors >= 0 && state, "adam_dev: bad argument");
  adam_advance_kernel<<<1, 1, 0, s>>>(state, lr0, decay_rate, decay_steps, beta1, beta2);
  CFN_LAUNCH_CHECK();
  return adam_update(n_tensors, params, grads, exp_avg, exp_avg_sq, numels, state, 0.f, 1.f, 1.f, beta1, beta2, eps,
                     grad_scale, s);
}

int launch_adam(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                float* const* exp_avg_sq, const int64_t* numels, float lr, float beta1, float beta2, float eps, int step,
                float grad_scale, cudaStream_t s) {
  CFN_CHECK_ARG(n_tensors >= 0 && step >= 1, "adam: bad argument");
  const float bc1 = 1.0f - powf(beta1, (float)step);
  const float bc2_sqrt = sqrtf(1.0f - powf(beta2, (float)step));
  return adam_update(n_tensors, params, grads, exp_avg, exp_avg_sq, numels, nullptr, lr, bc1, bc2_sqrt, beta1, beta2, eps,
                     grad_scale, s);
}

}  // namespace cfn
