// Hand-written update rules of the reference's net factory: networks.Sgd (DM/networks.py:354-371) and networks.Adam
// (DM/networks.py:374-420).  Arithmetic in fp32 with TF's operation order: every product, sum and quotient is rounded
// on its own (the __f*_rn intrinsics keep nvcc from contracting them into FMAs), the hyper-parameters are rounded to
// fp32 the way TF converts the Python floats, and (1 - b) is formed in double before that rounding (TF evaluates the
// Python expression first).
//
//   Sgd : delta = -lr * g
//   Adam: t' = t + 1 ; m' = b1*m + (1-b1)*g ; v' = b2*v + (1-b2)*(g*g)
//         delta = (-lr * (m' / (1 - b1^t'))) / (sqrt(v' / (1 - b2^t')) + eps)
//   x += delta (when asked)
//
// Adam state arena: [t, pad, pad, pad | m [n] | v [n]] (include/l2o_b200.h).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>

#include "l2o_internal.h"

namespace {

constexpr int kBlock = 256;
constexpr int kCoords = 3;    // coordinates a thread of the fused unroll keeps in registers (4 spills around the Adam divisions)
constexpr int kSeg = 512;     // steps per shared-memory segment of the fused unroll (fx partials + bias corrections)

struct Rule {
  float neg_lr, b1, omb1, b2, omb2, eps;
};

Rule make_rule(const l2o_rule_desc& d) {
  Rule r;
  r.neg_lr = (float)(-d.learning_rate);
  r.b1 = (float)d.beta1;
  r.omb1 = (float)(1.0 - d.beta1);
  r.b2 = (float)d.beta2;
  r.omb2 = (float)(1.0 - d.beta2);
  r.eps = (float)d.epsilon;
  return r;
}

// 1 - b^t' (_debias_adam_estimate, DM/networks.py:378-379): uniform over the coordinates of one step
__device__ __forceinline__ float debias(float b, float tp) { return __fsub_rn(1.0f, powf(b, tp)); }

// _update_adam_estimate + _debias_adam_estimate + the update of DM/networks.py:374-379,406-412
__device__ __forceinline__ float adam_coord(const Rule& r, float g, float& m, float& v, float c1, float c2) {
  m = __fadd_rn(__fmul_rn(r.b1, m), __fmul_rn(r.omb1, g));
  v = __fadd_rn(__fmul_rn(r.b2, v), __fmul_rn(r.omb2, __fmul_rn(g, g)));
  const float mh = __fdiv_rn(m, c1);
  const float vh = __fdiv_rn(v, c2);
  return __fdiv_rn(__fmul_rn(r.neg_lr, mh), __fadd_rn(__fsqrt_rn(vh), r.eps));
}

template <int KIND>
struct StepIO {
  const float* __restrict__ g;
  const float* __restrict__ m_in;
  const float* __restrict__ v_in;
  float* __restrict__ m_out;
  float* __restrict__ v_out;
  float* __restrict__ x;
  float* __restrict__ delta;

  __device__ __forceinline__ void one(const Rule& r, int64_t i, float c1, float c2) const {
    const float gi = __ldg(g + i);
    float d;
    if (KIND == L2O_RULE_ADAM) {
      float m = __ldg(m_in + i), v = __ldg(v_in + i);
      d = adam_coord(r, gi, m, v, c1, c2);
      m_out[i] = m;
      v_out[i] = v;
    } else {
      d = __fmul_rn(r.neg_lr, gi);
    }
    if (x) x[i] = __fadd_rn(x[i], d);
    if (delta) delta[i] = d;
  }

  // four coordinates starting at i (a multiple of 4; every pointer 16-byte aligned)
  __device__ __forceinline__ void four(const Rule& r, int64_t i, float c1, float c2) const {
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(g + i));
    float4 d4;
    if (KIND == L2O_RULE_ADAM) {
      float4 m4 = __ldg(reinterpret_cast<const float4*>(m_in + i));
      float4 v4 = __ldg(reinterpret_cast<const float4*>(v_in + i));
      d4.x = adam_coord(r, g4.x, m4.x, v4.x, c1, c2);
      d4.y = adam_coord(r, g4.y, m4.y, v4.y, c1, c2);
      d4.z = adam_coord(r, g4.z, m4.z, v4.z, c1, c2);
      d4.w = adam_coord(r, g4.w, m4.w, v4.w, c1, c2);
      *reinterpret_cast<float4*>(m_out + i) = m4;
      *reinterpret_cast<float4*>(v_out + i) = v4;
    } else {
      d4 = make_float4(__fmul_rn(r.neg_lr, g4.x), __fmul_rn(r.neg_lr, g4.y), __fmul_rn(r.neg_lr, g4.z),
                       __fmul_rn(r.neg_lr, g4.w));
    }
    if (x) {
      float4 x4 = *reinterpret_cast<const float4*>(x + i);
      x4 = make_float4(__fadd_rn(x4.x, d4.x), __fadd_rn(x4.y, d4.y), __fadd_rn(x4.z, d4.z), __fadd_rn(x4.w, d4.w));
      *reinterpret_cast<float4*>(x + i) = x4;
    }
    if (delta) *reinterpret_cast<float4*>(delta + i) = d4;
  }
};

// One rule step over n coordinates (grid-stride; memory-bound: Adam moves 28 B per coordinate).  The counter t is read
// from the state arena on the device, so a captured CUDA graph stays valid from replay to replay.
template <int KIND, bool VEC>
__global__ void __launch_bounds__(kBlock) rule_step_kernel(Rule r, int64_t n, StepIO<KIND> io,
                                                           const float* __restrict__ t_in, float* __restrict__ t_out) {
  float c1 = 1.0f, c2 = 1.0f;
  if (KIND == L2O_RULE_ADAM) {
    const float tp = __fadd_rn(*t_in, 1.0f);
    c1 = debias(r.b1, tp);
    c2 = debias(r.b2, tp);
    if (blockIdx.x == 0 && threadIdx.x < 4) t_out[threadIdx.x] = threadIdx.x == 0 ? tp : 0.0f;
  }
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (VEC) {
    const int64_t nv = n >> 2;
    for (int64_t i = i0; i < nv; i += stride) io.four(r, i << 2, c1, c2);
    i0 += nv << 2;
  }
  for (int64_t i = i0; i < n; i += stride) io.one(r, i, c1, c2);
}

// T rule steps over an in-kernel separable optimizee in one launch.  Every thread keeps kCoords coordinates (x, m, v
// and the optimizee constants) in registers across the steps of a segment; fx[t] is reduced per warp into shared
// memory and issued as one fp64 atomic per CTA per step.  The counter t is advanced by rule_counter_kernel afterwards
// (every CTA reads t before any could write it).
template <int KIND>
__global__ void __launch_bounds__(kBlock) rule_unroll_kernel(Rule r, int64_t n, int T, int opt_kind,
                                                             const float* __restrict__ oa, const float* __restrict__ ob,
                                                             float alpha, float fscale, float* __restrict__ x,
                                                             float* __restrict__ state, double* __restrict__ fx) {
  __shared__ double s_fx[kSeg];
  __shared__ float s_c1[kSeg], s_c2[kSeg];
  const float t0 = KIND == L2O_RULE_ADAM ? state[0] : 0.0f;
  float* __restrict__ mg = state + 4;
  float* __restrict__ vg = state + 4 + n;
  const int64_t threads = (int64_t)gridDim.x * kBlock;
  const int64_t per_round = threads * kCoords;
  const int64_t rounds = (n + per_round - 1) / per_round;
  const int64_t base = (int64_t)blockIdx.x * kBlock + threadIdx.x;
  const int lane = threadIdx.x & 31;
  for (int s0 = 0; s0 <= T; s0 += kSeg) {
    const int s1 = min(s0 + kSeg, T + 1);   // step indices [s0, s1): t < T evaluates and updates, t == T evaluates
    for (int i = threadIdx.x; i < s1 - s0; i += kBlock) {
      s_fx[i] = 0.0;
      if (KIND == L2O_RULE_ADAM) {
        const float tp = __fadd_rn(t0, (float)(s0 + i + 1));
        s_c1[i] = debias(r.b1, tp);
        s_c2[i] = debias(r.b2, tp);
      }
    }
    __syncthreads();
    for (int64_t rd = 0; rd < rounds; ++rd) {
      float xr[kCoords], mr[kCoords], vr[kCoords], ar[kCoords], br[kCoords];
      bool ok[kCoords];
#pragma unroll
      for (int k = 0; k < kCoords; ++k) {
        const int64_t i = rd * per_round + k * threads + base;
        ok[k] = i < n;
        xr[k] = ok[k] ? x[i] : 0.0f;
        ar[k] = ok[k] ? __ldg(oa + i) : 0.0f;
        br[k] = ok[k] ? __ldg(ob + i) : 0.0f;
        mr[k] = (KIND == L2O_RULE_ADAM && ok[k]) ? mg[i] : 0.0f;
        vr[k] = (KIND == L2O_RULE_ADAM && ok[k]) ? vg[i] : 0.0f;
      }
      for (int t = s0; t < s1; ++t) {
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < kCoords; ++k) {
          if (!ok[k]) continue;
          float f, g;
          l2o::optimizee_eval(opt_kind, xr[k], ar[k], br[k], alpha, fscale, f, g);
          acc += (double)f;
          if (t < T) {
            const float d = KIND == L2O_RULE_ADAM ? adam_coord(r, g, mr[k], vr[k], s_c1[t - s0], s_c2[t - s0])
                                                  : __fmul_rn(r.neg_lr, g);
            xr[k] = __fadd_rn(xr[k], d);
          }
        }
        acc = l2o::warp_sum_d(acc);
        if (lane == 0) atomicAdd(&s_fx[t - s0], acc);
      }
#pragma unroll
      for (int k = 0; k < kCoords; ++k) {
        const int64_t i = rd * per_round + k * threads + base;
        if (!ok[k]) continue;
        x[i] = xr[k];
        if (KIND == L2O_RULE_ADAM) {
          mg[i] = mr[k];
          vg[i] = vr[k];
        }
      }
    }
    __syncthreads();
    if (fx)
      for (int i = threadIdx.x; i < s1 - s0; i += kBlock) atomicAdd(&fx[s0 + i], s_fx[i]);
    __syncthreads();
  }
}

__global__ void rule_counter_kernel(float* state, int T) { state[0] = __fadd_rn(state[0], (float)T); }

bool aligned16(const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

bool desc_ok(const l2o_rule_desc* d) {
  if (!d || (d->kind != L2O_RULE_SGD && d->kind != L2O_RULE_ADAM)) return false;
  if (!(d->learning_rate >= 0.0)) return false;
  if (d->kind == L2O_RULE_ADAM && !(d->beta1 >= 0.0 && d->beta1 < 1.0 && d->beta2 >= 0.0 && d->beta2 < 1.0))
    return false;
  return true;
}

template <int KIND>
int launch_step(const Rule& r, const l2o_rule_step_args& a, cudaStream_t st) {
  const int64_t n = a.n;
  StepIO<KIND> io{a.g, nullptr, nullptr, nullptr, nullptr, a.x, a.delta};
  const float* t_in = nullptr;
  float* t_out = nullptr;
  if (KIND == L2O_RULE_ADAM) {
    t_in = a.state_in;
    t_out = a.state_out;
    io.m_in = a.state_in + 4;
    io.v_in = a.state_in + 4 + n;
    io.m_out = a.state_out + 4;
    io.v_out = a.state_out + 4 + n;
  }
  const bool vec = aligned16(io.g) && aligned16(io.m_in) && aligned16(io.v_in) && aligned16(io.m_out) &&
                   aligned16(io.v_out) && aligned16(io.x) && aligned16(io.delta);
  const int sms = l2o::device_sms();
  if (sms <= 0) return l2o::set_cuda_error(cudaGetLastError(), "cudaDeviceGetAttribute");
  const int64_t work = vec ? (n >> 2) + (n & 3) : n;
  // at least one CTA: an Adam step over no coordinate still advances the counter
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((work + kBlock - 1) / kBlock, (int64_t)sms * 8));
  if (vec)
    rule_step_kernel<KIND, true><<<blocks, kBlock, 0, st>>>(r, n, io, t_in, t_out);
  else
    rule_step_kernel<KIND, false><<<blocks, kBlock, 0, st>>>(r, n, io, t_in, t_out);
  l2o::count_launch();
  L2O_CUDA_TRY(cudaGetLastError());
  return L2O_OK;
}

template <int KIND>
int launch_unroll(const Rule& r, const l2o_rule_unroll_args& a, cudaStream_t st) {
  const int sms = l2o::device_sms();
  if (sms <= 0) return l2o::set_cuda_error(cudaGetLastError(), "cudaDeviceGetAttribute");
  int per_sm = 0;
  L2O_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rule_unroll_kernel<KIND>, kBlock, 0));
  // every CTA resident at once; fewer when n is small (a CTA covers kBlock coordinates per register slot)
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((a.n + kBlock - 1) / kBlock,
                                                                  (int64_t)sms * std::max(per_sm, 1)));
  rule_unroll_kernel<KIND><<<blocks, kBlock, 0, st>>>(r, a.n, a.T, a.opt_kind, a.opt_a, a.opt_b, a.opt_alpha,
                                                      a.opt_fscale, a.x, a.state, a.fx);
  l2o::count_launch();
  L2O_CUDA_TRY(cudaGetLastError());
  if (KIND == L2O_RULE_ADAM && a.T > 0) {
    rule_counter_kernel<<<1, 1, 0, st>>>(a.state, a.T);
    l2o::count_launch();
    L2O_CUDA_TRY(cudaGetLastError());
  }
  return L2O_OK;
}

}  // namespace

extern "C" {

int l2o_rule_state_floats(const l2o_rule_desc* d, int64_t n, int64_t* out) {
  if (!desc_ok(d) || n < 0 || !out) return L2O_E_INVALID;
  *out = d->kind == L2O_RULE_ADAM ? 4 + 2 * n : 0;
  return L2O_OK;
}

int l2o_rule_step(const l2o_rule_desc* d, const l2o_rule_step_args* a, void* stream) {
  if (!desc_ok(d) || !a || a->n < 0 || !a->g) return L2O_E_INVALID;
  if (d->kind == L2O_RULE_ADAM) {
    if (!a->state_in || !a->state_out) return L2O_E_INVALID;
    // the counter of state_in is read by every CTA while CTA 0 writes state_out's: the arenas must not overlap
    const uintptr_t in0 = reinterpret_cast<uintptr_t>(a->state_in), out0 = reinterpret_cast<uintptr_t>(a->state_out);
    const uintptr_t bytes = (uintptr_t)(4 + 2 * a->n) * sizeof(float);
    if (in0 < out0 + bytes && out0 < in0 + bytes) return L2O_E_INVALID;
  }
  if (a->n == 0 && d->kind == L2O_RULE_SGD) return L2O_OK;
  const Rule r = make_rule(*d);
  cudaStream_t st = (cudaStream_t)stream;
  return d->kind == L2O_RULE_ADAM ? launch_step<L2O_RULE_ADAM>(r, *a, st) : launch_step<L2O_RULE_SGD>(r, *a, st);
}

int l2o_rule_unroll_fwd(const l2o_rule_desc* d, const l2o_rule_unroll_args* a, void* stream) {
  if (!desc_ok(d) || !a || a->n < 0 || a->T < 0) return L2O_E_INVALID;
  if (a->opt_kind < L2O_OPT_NONE || a->opt_kind > L2O_OPT_QUADRATIC_BATCH) return L2O_E_INVALID;
  if (a->opt_kind != L2O_OPT_RASTRIGIN_SEP && a->opt_kind != L2O_OPT_QUADRATIC_DIAG) return L2O_E_UNSUPPORTED;
  if (!a->x || !a->opt_a || !a->opt_b) return L2O_E_INVALID;
  if (d->kind == L2O_RULE_ADAM && !a->state) return L2O_E_INVALID;
  if (a->n == 0) return L2O_OK;
  const Rule r = make_rule(*d);
  cudaStream_t st = (cudaStream_t)stream;
  return d->kind == L2O_RULE_ADAM ? launch_unroll<L2O_RULE_ADAM>(r, *a, st) : launch_unroll<L2O_RULE_SGD>(r, *a, st);
}

}  // extern "C"
