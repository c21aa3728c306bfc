// The optimizer tail of the train steps (SURVEY.md 8f-3): multi-tensor Adam / AdamW over ONE flat fp32 buffer that holds
// every live parameter, its flat gradient twin right after the gradient all-reduce, and the global-norm clip of DAG-ERC.
//   reference: torch.optim.Adam(lr 1e-4, weight_decay 1e-8)   track_mm/cogmen.py:50,187-189 (dgcn.py:41, mmgcn.py:34)
//              torch.optim.AdamW + clip_grad_norm_(5)           track_mm/dagerc.py:39,229-231
// Everything a step needs lives on the device (step counter, squared norm), so the whole train step -- graph build,
// forward, backward, all-reduce, optimizer -- can be captured in one CUDA graph and replayed without host arithmetic.
#include "common.cuh"

namespace ercg {

// fixed-order two-level reduction of sum x^2 (fp64 partials): bit-reproducible, no atomics
__global__ void __launch_bounds__(256) sumsq_partial_kernel(const float* __restrict__ x, long long n, double* __restrict__ part) {
  __shared__ double sm[8];
  double acc = 0.0;
  const long long stride = (long long)gridDim.x * 256;
  const long long n4 = aligned16(x) ? (n >> 2) : 0;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += stride) {
    const float4 v = ld4(x + 4 * i);
    acc += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += stride) acc += (double)x[i] * x[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += sm[w];
    part[blockIdx.x] = t;
  }
}
__global__ void sumsq_final_kernel(const double* __restrict__ part, int nb, float* __restrict__ out) {
  double a = 0.0;
  for (int i = threadIdx.x; i < nb; i += 32) a += part[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  if (threadIdx.x == 0) out[0] = (float)a;
}

struct AdamArgs {
  float* p; const float* g; float* m; float* v; long long n;
  float lr, beta1, beta2, eps, weight_decay; int decoupled;
  float grad_scale;             // multiplies every gradient (1/world for an averaged all-reduce, 1 otherwise)
  const float* sumsq; float max_norm;   // optional clip_grad_norm_: coefficient min(1, max_norm / (sqrt(sumsq) * grad_scale + 1e-6))
  long long* step;              // device step counter, incremented by this launch (bias correction uses the new value)
};

__device__ __forceinline__ float adam_one(float p, float g, float& m, float& v, const AdamArgs& a, float gs, float c1, float c2s) {
  g *= gs;
  if (a.decoupled) p *= 1.0f - a.lr * a.weight_decay;          // AdamW: param.mul_(1 - lr * wd)
  else if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);   // Adam: grad.add(param, alpha=wd)
  m = m + (g - m) * (1.0f - a.beta1);                          // exp_avg.lerp_(grad, 1 - beta1)
  v = a.beta2 * v + (1.0f - a.beta2) * g * g;                  // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
  const float denom = sqrtf(v) / c2s + a.eps;                  // (exp_avg_sq.sqrt() / sqrt(bias_correction2)).add_(eps)
  return p - (a.lr / c1) * (m / denom);                        // param.addcdiv_(exp_avg, denom, value=-lr / bias_correction1)
}

// GUARDED (ercg_adam_step_guarded): every thread returns before touching p, m, v when *skip != 0 -- the status word of a
// peer-memory exchange that timed out, so a garbage-summed gradient is never applied.  The arithmetic is the same either way.
template <bool GUARDED>
__global__ void __launch_bounds__(256) adam_kernel(AdamArgs a, const int* __restrict__ skip) {
  if (GUARDED && *skip != 0) return;
  const long long t = a.step[0] + 1;                           // the counter is bumped by a SEPARATE launch after this one
  const float c1 = (float)(1.0 - pow((double)a.beta1, (double)t));          // bias corrections in double, like torch.optim
  const float c2s = (float)sqrt(1.0 - pow((double)a.beta2, (double)t));
  float gs = a.grad_scale;
  if (a.sumsq) {
    const float norm = sqrtf(a.sumsq[0]) * a.grad_scale;
    const float coef = a.max_norm / (norm + 1e-6f);            // torch.nn.utils.clip_grad_norm_
    gs *= coef < 1.0f ? coef : 1.0f;
  }
  const long long stride = (long long)gridDim.x * 256;
  const bool vec = aligned16(a.p) && aligned16(a.g) && aligned16(a.m) && aligned16(a.v);
  const long long n4 = vec ? (a.n >> 2) : 0;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += stride) {
    float4 p = ld4(a.p + 4 * i), m = ld4(a.m + 4 * i), v = ld4(a.v + 4 * i);
    const float4 g = ld4(a.g + 4 * i);
    p.x = adam_one(p.x, g.x, m.x, v.x, a, gs, c1, c2s);
    p.y = adam_one(p.y, g.y, m.y, v.y, a, gs, c1, c2s);
    p.z = adam_one(p.z, g.z, m.z, v.z, a, gs, c1, c2s);
    p.w = adam_one(p.w, g.w, m.w, v.w, a, gs, c1, c2s);
    st4(a.p + 4 * i, p); st4(a.m + 4 * i, m); st4(a.v + 4 * i, v);
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * 256 + threadIdx.x; i < a.n; i += stride) {
    float m = a.m[i], v = a.v[i];
    a.p[i] = adam_one(a.p[i], a.g[i], m, v, a, gs, c1, c2s);
    a.m[i] = m; a.v[i] = v;
  }
}
// separate single-thread launch: bumping the counter inside adam_kernel would race with blocks that have not read it yet
template <bool GUARDED>
__global__ void step_bump_kernel(long long* step, const int* __restrict__ skip) {
  if (GUARDED && *skip != 0) return;
  step[0] += 1;
}

template <bool GUARDED>
int adam_launch(const AdamArgs& a, const int* skip, cudaStream_t stream) {
  if (a.n > 0) {
    long long want = (a.n / 4 + 255) / 256;
    const long long cap = 8LL * device_sm_count();
    const int nb = (int)(want < 1 ? 1 : (want > cap ? cap : want));
    adam_kernel<GUARDED><<<nb, 256, 0, stream>>>(a, skip);
    int rc = finish_launch();
    if (rc) return rc;
  }
  step_bump_kernel<GUARDED><<<1, 1, 0, stream>>>(a.step, skip);
  return finish_launch();
}

int adam_args(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
              float weight_decay, int decoupled, float grad_scale, const float* sumsq, float max_norm, int64_t* step_dev,
              AdamArgs* a) {
  if (n < 0 || !step_dev) return ERCG_EINVAL;
  if (n > 0 && (!p || !g || !m || !v)) return ERCG_EINVAL;
  if (!(beta1 >= 0.f && beta1 < 1.f) || !(beta2 >= 0.f && beta2 < 1.f) || !(eps >= 0.f)) return ERCG_EINVAL;
  *a = AdamArgs{p, g, m, v, (long long)n, lr, beta1, beta2, eps, weight_decay, decoupled, grad_scale, sumsq, max_norm,
                reinterpret_cast<long long*>(step_dev)};
  return ERCG_OK;
}

}  // namespace ercg

using namespace ercg;

extern "C" size_t ercg_sumsq_workspace_bytes(int64_t n) {
  (void)n;
  return sizeof(double) * 1024;
}

extern "C" int ercg_sumsq(const float* x, int64_t n, float* out, void* workspace, size_t workspace_bytes, void* stream) {
  if (n < 0 || !out) return ERCG_EINVAL;
  if (!workspace || workspace_bytes < ercg_sumsq_workspace_bytes(n)) return ERCG_EWORKSPACE;
  if (n > 0 && !x) return ERCG_EINVAL;
  long long want = (n / 4 + 255) / 256;
  const int nb = (int)(want < 1 ? 1 : (want > 1024 ? 1024 : want));
  sumsq_partial_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(x, n, reinterpret_cast<double*>(workspace));
  int rc = finish_launch();
  if (rc) return rc;
  sumsq_final_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(reinterpret_cast<const double*>(workspace), nb, out);
  return finish_launch();
}

extern "C" int ercg_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                              float eps, float weight_decay, int decoupled, float grad_scale, const float* sumsq,
                              float max_norm, int64_t* step_dev, void* stream) {
  AdamArgs a;
  const int rc = adam_args(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, decoupled, grad_scale, sumsq, max_norm, step_dev, &a);
  return rc ? rc : adam_launch<false>(a, nullptr, (cudaStream_t)stream);
}

// The data-parallel trainer's step after a peer-memory gradient all-reduce (train_mm.py under torchrun): skip_if_nonzero is
// that communicator's sticky status word (ercg_p2p_status_word), so once an exchange has timed out no update is applied.
extern "C" int ercg_adam_step_guarded(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                                      float beta2, float eps, float weight_decay, int decoupled, float grad_scale,
                                      const float* sumsq, float max_norm, int64_t* step_dev, void* stream,
                                      const int* skip_if_nonzero) {
  if (!skip_if_nonzero) return ERCG_EINVAL;
  AdamArgs a;
  const int rc = adam_args(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, decoupled, grad_scale, sumsq, max_norm, step_dev, &a);
  return rc ? rc : adam_launch<true>(a, skip_if_nonzero, (cudaStream_t)stream);
}
