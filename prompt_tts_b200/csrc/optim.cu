// Optimiser kernels: sums of squares for the gradient norm (atomic, and per-block partials for the deterministic norm), AdamW
// (host-side coefficients, and the graph-safe variant with device-resident state, a bf16 shadow write and the EMA update), and the
// EMA bookkeeping and master <-> EMA swap.
#include "common.cuh"

namespace {

__global__ void sumsq_kernel(const float* __restrict__ x, long long n, float* __restrict__ out) {
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) acc += x[i] * x[i];
  acc = block_sum(acc);
  if (threadIdx.x == 0) atomicAdd(out, acc);
}

__global__ void sumsq_bf16_kernel(const bf16* __restrict__ x, long long n8, float* __restrict__ out) {
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float f[8];
    load8(x + i * 8, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) acc = fmaf(f[j], f[j], acc);
  }
  acc = block_sum(acc);
  if (threadIdx.x == 0) atomicAdd(out, acc);
}

__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
                             float lr, float b1, float b2, float eps, float wd, float bc1, float bc2, const float* __restrict__ gnorm_sq,
                             float max_norm, float gscale) {
  float clip = gscale;
  if (gnorm_sq && max_norm > 0.f) {
    const float norm = sqrtf(*gnorm_sq) * gscale;
    clip *= fminf(1.f, max_norm / (norm + 1e-6f));
  }
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * clip;
    float pi = p[i] * (1.f - lr * wd);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / sqrtf(bc2) + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}

// ---- graph-safe optimiser state: everything that changes from step to step lives in device memory, so one captured step replays
// correctly.  `st` = PT_OPT_STATE_FLOATS fp32 words (see include/prompt_tts_b200.h): hyper-parameters written by the host (or by an LR
// scheduler, at any time), the step counter incremented HERE, and the per-step coefficients the elementwise kernel reads.
// Deterministic global norm: every block writes ONE partial sum of squares (fixed block -> element mapping, fixed in-block tree),
// and the coefficient kernel adds the partials in a fixed order.  Atomic accumulation would round differently from run to run -- and
// from rank to rank: data-parallel replicas that clip by norms differing in the last bit drift apart, which DDP + clip_grad_norm_
// in the reference never do.
template <bool IN_BF16>
__global__ void __launch_bounds__(256) sumsq_partials_kernel(const void* __restrict__ xv, long long n, float* __restrict__ partials) {
  float acc = 0.f;
  if (IN_BF16) {
    const bf16* x = reinterpret_cast<const bf16*>(xv);
    const long long n8 = n >> 3;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
      float f[8];
      load8(x + i * 8, f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc = fmaf(f[j], f[j], acc);
    }
  } else {
    const float4* x = reinterpret_cast<const float4*>(xv);
    const long long n4 = n >> 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
      const float4 t = x[i];
      acc = fmaf(t.x, t.x, acc), acc = fmaf(t.y, t.y, acc), acc = fmaf(t.z, t.z, acc), acc = fmaf(t.w, t.w, acc);
    }
  }
  acc = warp_sum(acc);
  __shared__ float sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) v += sh[w];
    partials[blockIdx.x] = v;
  }
}

__global__ void adamw_prepare_kernel(float* __restrict__ st, const float* __restrict__ gnorm_sq, const float* __restrict__ partials, int nparts) {
  __shared__ float tot;
  if (partials != nullptr) {      // fixed-order sum of the per-block partials: lane l adds l, l + 32, ...; then the shuffle tree
    float a = 0.f;
    for (int i = threadIdx.x; i < nparts; i += 32) a += partials[i];
    a = warp_sum(a);
    if (threadIdx.x == 0) tot = a;
  } else if (threadIdx.x == 0) {
    tot = gnorm_sq != nullptr ? *gnorm_sq : -1.f;
  }
  __syncwarp();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const float sumsq = tot;
  const float lr = st[PT_OPT_LR], b1 = st[PT_OPT_BETA1], b2 = st[PT_OPT_BETA2], wd = st[PT_OPT_WD], max_norm = st[PT_OPT_MAX_NORM],
              gscale = st[PT_OPT_GSCALE];
  const int step = __float_as_int(st[PT_OPT_STEP]) + 1;
  st[PT_OPT_STEP] = __int_as_float(step);
  // torch.optim.AdamW: bias_correction = 1 - beta ** step (python doubles)
  const double bc1 = 1.0 - pow((double)b1, (double)step), bc2 = 1.0 - pow((double)b2, (double)step);
  float clip = gscale;
  float norm = 0.f;
  if (sumsq >= 0.f) {
    norm = sqrtf(sumsq) * gscale;
    if (max_norm > 0.f) clip *= fminf(1.f, max_norm / (norm + 1e-6f));   // torch.nn.utils.clip_grad_norm_
  }
  st[PT_OPT_GNORM_SQ] = fmaxf(sumsq, 0.f);
  st[PT_OPT_CLIP] = clip;
  st[PT_OPT_STEP_SIZE] = (float)((double)lr / bc1);
  st[PT_OPT_INV_SQRT_BC2] = (float)(1.0 / sqrt(bc2));
  st[PT_OPT_DECAY] = 1.f - lr * wd;
  st[PT_OPT_GNORM] = norm;
}

// p, g, m, v fp32 flat buffers in one common layout; w (optional) the bf16 shadow of p in the same layout: the GEMM operands are
// views of it, so the updated weights need no re-pack pass.  4 elements per thread per iteration (n % 4 == 0).
// EMA: e (same layout) = e - c * (e - p_new) with c = float(1 - decay) from pt_ema_prepare; the update costs 8 bytes per element
// here against 12 in a pass of its own.  The EMA arguments come last so that the two plain instantiations keep their code.
template <bool G_BF16, bool EMA>
__global__ void __launch_bounds__(256) adamw_dev_kernel(float* __restrict__ p, const void* __restrict__ gv, float* __restrict__ m,
                                                        float* __restrict__ v, bf16* __restrict__ w, long long n4,
                                                        const float* __restrict__ st, float* __restrict__ e,
                                                        const double* __restrict__ est) {
  const float clip = st[PT_OPT_CLIP], step_size = st[PT_OPT_STEP_SIZE], isb2 = st[PT_OPT_INV_SQRT_BC2], decay = st[PT_OPT_DECAY];
  const float b1 = st[PT_OPT_BETA1], b2 = st[PT_OPT_BETA2], eps = st[PT_OPT_EPS];
  const float c = EMA ? (float)est[PT_EMA_COEF] : 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 pi = reinterpret_cast<const float4*>(p)[i];
    float4 mi = reinterpret_cast<const float4*>(m)[i];
    float4 vi = reinterpret_cast<const float4*>(v)[i];
    float4 ei;
    if (EMA) ei = reinterpret_cast<const float4*>(e)[i];
    float gi[4];
    if (G_BF16) {
      const uint2 t = reinterpret_cast<const uint2*>(gv)[i];
      const float2 a = bf2_to_f2(t.x), b = bf2_to_f2(t.y);
      gi[0] = a.x, gi[1] = a.y, gi[2] = b.x, gi[3] = b.y;
    } else {
      const float4 t = reinterpret_cast<const float4*>(gv)[i];
      gi[0] = t.x, gi[1] = t.y, gi[2] = t.z, gi[3] = t.w;
    }
    float pp[4] = {pi.x, pi.y, pi.z, pi.w}, mm[4] = {mi.x, mi.y, mi.z, mi.w}, vv[4] = {vi.x, vi.y, vi.z, vi.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float g = gi[j] * clip;
      const float pd = pp[j] * decay;
      mm[j] = b1 * mm[j] + (1.f - b1) * g;
      vv[j] = b2 * vv[j] + (1.f - b2) * g * g;
      const float denom = sqrtf(vv[j]) * isb2 + eps;
      pp[j] = pd - step_size * (mm[j] / denom);
    }
    reinterpret_cast<float4*>(p)[i] = make_float4(pp[0], pp[1], pp[2], pp[3]);
    reinterpret_cast<float4*>(m)[i] = make_float4(mm[0], mm[1], mm[2], mm[3]);
    reinterpret_cast<float4*>(v)[i] = make_float4(vv[0], vv[1], vv[2], vv[3]);
    if (w != nullptr) reinterpret_cast<uint2*>(w)[i] = make_uint2(f2_to_bf2(pp[0], pp[1]), f2_to_bf2(pp[2], pp[3]));
    if (EMA) {      // diffusers: s_param.sub_(one_minus_decay * (s_param - param)), three fp32 roundings
      float ee[4] = {ei.x, ei.y, ei.z, ei.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) ee[j] = __fsub_rn(ee[j], __fmul_rn(c, __fsub_rn(ee[j], pp[j])));
      reinterpret_cast<float4*>(e)[i] = make_float4(ee[0], ee[1], ee[2], ee[3]);
    }
  }
}

// diffusers 0.15 EMAModel.step's bookkeeping and get_decay, in its order and in double precision (python floats)
__global__ void ema_prepare_kernel(double* __restrict__ st) {
  const double opt_step = st[PT_EMA_STEP] + 1.0;
  st[PT_EMA_STEP] = opt_step;
  const double step = fmax(0.0, opt_step - st[PT_EMA_UPDATE_AFTER] - 1.0);
  double decay = 0.0;
  if (step > 0.0) {
    decay = st[PT_EMA_USE_WARMUP] != 0.0 ? 1.0 - pow(1.0 + step / st[PT_EMA_INV_GAMMA], -st[PT_EMA_POWER]) : (1.0 + step) / (10.0 + step);
    decay = fmax(fmin(decay, st[PT_EMA_DECAY]), st[PT_EMA_MIN_DECAY]);
  }
  st[PT_EMA_CUR_DECAY] = decay;
  st[PT_EMA_COEF] = (double)(float)(1.0 - decay);
}

// master <-> EMA exchange; the GEMM operands (w = bf16 shadow of p) follow the new p
__global__ void ema_swap_kernel(float4* __restrict__ p, float4* __restrict__ e, uint2* __restrict__ w, long long n4) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 a = p[i], b = e[i];
    p[i] = b;
    e[i] = a;
    w[i] = make_uint2(f2_to_bf2(b.x, b.y), f2_to_bf2(b.z, b.w));
  }
}

}  // namespace

#define ST ((cudaStream_t)stream)

extern "C" int pt_sumsq_f32(const float* x, int64_t n, float* out, void* stream) {
  PT_REQUIRE(n > 0, "sumsq: n=%lld", (long long)n);
  sumsq_kernel<<<grid_for(n, 1024, 4), 256, 0, ST>>>(x, n, out);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_sumsq_bf16(const void* x, int64_t n, float* out, void* stream) {
  PT_REQUIRE(n > 0 && n % 8 == 0, "sumsq_bf16: n=%lld must be a positive multiple of 8", (long long)n);
  sumsq_bf16_kernel<<<grid_for(n / 8, 1024, 4), 256, 0, ST>>>((const bf16*)x, n / 8, out);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps, float wd,
                             int step, const float* gnorm_sq, float max_norm, float gscale, void* stream) {
  PT_REQUIRE(n > 0 && step >= 1, "adamw: n=%lld step=%d", (long long)n, step);
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  adamw_kernel<<<grid_for(n, 1024, 4), 256, 0, ST>>>(p, g, m, v, n, lr, beta1, beta2, eps, wd, bc1, bc2, gnorm_sq, max_norm, gscale);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_adamw_prepare(float* state, const float* gnorm_sq, void* stream) {
  PT_REQUIRE(state != nullptr, "adamw_prepare: null state");
  adamw_prepare_kernel<<<1, 32, 0, ST>>>(state, gnorm_sq, nullptr, 0);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_sumsq_partials(const void* x, int x_is_bf16, int64_t n, float* partials, int nparts, void* stream) {
  PT_REQUIRE(n > 0 && n % 8 == 0 && nparts >= 1 && nparts <= 65535, "sumsq_partials: n=%lld (multiple of 8) nparts=%d", (long long)n, nparts);
  if (x_is_bf16) sumsq_partials_kernel<true><<<nparts, 256, 0, ST>>>(x, n, partials);
  else sumsq_partials_kernel<false><<<nparts, 256, 0, ST>>>(x, n, partials);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_adamw_prepare_det(float* state, const float* partials, int nparts, void* stream) {
  PT_REQUIRE(state != nullptr && partials != nullptr && nparts >= 1, "adamw_prepare_det: null pointer");
  adamw_prepare_kernel<<<1, 32, 0, ST>>>(state, nullptr, partials, nparts);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
template <bool EMA>
static int adamw_dev_launch(float* p, const void* g, int g_is_bf16, float* m, float* v, void* w_bf16, int64_t n, const float* state,
                            float* ema, const double* ema_state, cudaStream_t st) {
  const unsigned grid = grid_for(n / 4, 1024, 4);
  if (g_is_bf16) adamw_dev_kernel<true, EMA><<<grid, 256, 0, st>>>(p, g, m, v, (bf16*)w_bf16, n / 4, state, ema, ema_state);
  else adamw_dev_kernel<false, EMA><<<grid, 256, 0, st>>>(p, g, m, v, (bf16*)w_bf16, n / 4, state, ema, ema_state);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_adamw_step_dev(float* p, const void* g, int g_is_bf16, float* m, float* v, void* w_bf16, int64_t n, const float* state,
                                 void* stream) {
  PT_REQUIRE(n > 0 && n % 4 == 0, "adamw_step_dev: n=%lld must be a positive multiple of 4", (long long)n);
  PT_REQUIRE(p && g && m && v && state, "adamw_step_dev: null pointer");
  return adamw_dev_launch<false>(p, g, g_is_bf16, m, v, w_bf16, n, state, nullptr, nullptr, ST);
}
extern "C" int pt_ema_prepare(double* ema_state, void* stream) {
  PT_REQUIRE(ema_state != nullptr, "ema_prepare: null state");
  ema_prepare_kernel<<<1, 1, 0, ST>>>(ema_state);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_adamw_ema_step_dev(float* p, const void* g, int g_is_bf16, float* m, float* v, void* w_bf16, float* ema, int64_t n,
                                     const float* state, const double* ema_state, void* stream) {
  PT_REQUIRE(n > 0 && n % 4 == 0, "adamw_ema_step_dev: n=%lld must be a positive multiple of 4", (long long)n);
  PT_REQUIRE(p && g && m && v && ema && state && ema_state, "adamw_ema_step_dev: null pointer");
  return adamw_dev_launch<true>(p, g, g_is_bf16, m, v, w_bf16, n, state, ema, ema_state, ST);
}
extern "C" int pt_ema_swap(float* p, float* ema, void* w_bf16, int64_t n, void* stream) {
  PT_REQUIRE(n > 0 && n % 4 == 0, "ema_swap: n=%lld must be a positive multiple of 4", (long long)n);
  PT_REQUIRE(p && ema && w_bf16, "ema_swap: null pointer");
  ema_swap_kernel<<<grid_for(n / 4, 1024, 4), 256, 0, ST>>>((float4*)p, (float4*)ema, (uint2*)w_bf16, n / 4);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
