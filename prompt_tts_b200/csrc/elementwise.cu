// Bandwidth-bound pieces: softmax fwd/bwd, GEGLU fwd/bwd, adds, casts, copies, up-sampling, layout
// changes, weight packing, column sums, timestep sinusoid, text embedding (the train step's loss and the samplers' steps are in
// diffusion.cu, the optimiser in optim.cu).  All: 16-byte vector accesses where the layout allows, grid sized in multiples of the SM count.
#include "common.cuh"

namespace {

// ------------------------------------------------------------------------------------------------ softmax
constexpr int SM_MAXV = 16;  // 16 float4 per lane -> n <= 2048

__global__ void softmax_fwd_kernel(const float* __restrict__ S, bf16* __restrict__ P, long long rows, int n, long long ld_s, long long ld_p) {
  const int lane = threadIdx.x & 31;
  const long long wstride = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows; row += wstride) {
    const float* s = S + row * ld_s;
    float4 v[SM_MAXV];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < SM_MAXV; ++i) {
      const int j = (lane + i * 32) * 4;
      if (j < n) {
        v[i] = *reinterpret_cast<const float4*>(s + j);
        if (j + 1 >= n) v[i].y = -INFINITY;
        if (j + 2 >= n) v[i].z = -INFINITY;
        if (j + 3 >= n) v[i].w = -INFINITY;
        mx = fmaxf(mx, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w)));
      }
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < SM_MAXV; ++i) {
      const int j = (lane + i * 32) * 4;
      if (j < n) {
        v[i].x = __expf(v[i].x - mx);
        v[i].y = __expf(v[i].y - mx);
        v[i].z = __expf(v[i].z - mx);
        v[i].w = __expf(v[i].w - mx);
        sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
      }
    }
    const float inv = 1.f / warp_sum(sum);
    bf16* p = P + row * ld_p;
#pragma unroll
    for (int i = 0; i < SM_MAXV; ++i) {
      const int j = (lane + i * 32) * 4;
      if (j < n) {
        __nv_bfloat162 a = __floats2bfloat162_rn(v[i].x * inv, v[i].y * inv);
        __nv_bfloat162 b = __floats2bfloat162_rn(v[i].z * inv, v[i].w * inv);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&a);
        u.y = *reinterpret_cast<uint32_t*>(&b);
        *reinterpret_cast<uint2*>(p + j) = u;  // pad columns (>= n) hold zeros: exp(-inf)
      }
    }
  }
}

__global__ void softmax_bwd_kernel(const float* __restrict__ dP, const bf16* __restrict__ P, bf16* __restrict__ dS, long long rows, int n,
                                   long long ld_s, long long ld_p, float scale) {
  const int lane = threadIdx.x & 31;
  const long long wstride = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < rows; row += wstride) {
    const float* dp = dP + row * ld_s;
    const bf16* p = P + row * ld_p;
    float4 g[SM_MAXV], pr[SM_MAXV];
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < SM_MAXV; ++i) {
      const int j = (lane + i * 32) * 4;
      if (j < n) {
        g[i] = *reinterpret_cast<const float4*>(dp + j);
        const uint2 u = *reinterpret_cast<const uint2*>(p + j);
        const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
        const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
        pr[i] = make_float4(a.x, a.y, b.x, b.y);
        if (j + 1 >= n) pr[i].y = 0.f, g[i].y = 0.f;
        if (j + 2 >= n) pr[i].z = 0.f, g[i].z = 0.f;
        if (j + 3 >= n) pr[i].w = 0.f, g[i].w = 0.f;
        dot += g[i].x * pr[i].x + g[i].y * pr[i].y + g[i].z * pr[i].z + g[i].w * pr[i].w;
      }
    }
    dot = warp_sum(dot);
    bf16* o = dS + row * ld_p;
#pragma unroll
    for (int i = 0; i < SM_MAXV; ++i) {
      const int j = (lane + i * 32) * 4;
      if (j < n) {
        __nv_bfloat162 a = __floats2bfloat162_rn(scale * pr[i].x * (g[i].x - dot), scale * pr[i].y * (g[i].y - dot));
        __nv_bfloat162 b = __floats2bfloat162_rn(scale * pr[i].z * (g[i].z - dot), scale * pr[i].w * (g[i].w - dot));
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&a);
        u.y = *reinterpret_cast<uint32_t*>(&b);
        *reinterpret_cast<uint2*>(o + j) = u;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ GEGLU
// erf by Abramowitz & Stegun 7.1.26 (|error| <= 1.5e-7, the accuracy class of erff itself): one reciprocal, one exponential and
// five FMAs instead of erff's branchy ~25-instruction polynomial -- the GEGLU kernels were issue-bound on it (ncu: 76 % issue
// slots busy at 40-50 % of HBM bandwidth).  The exponential is exp(-g^2/2), which is also the Gaussian factor of the derivative.
__device__ __forceinline__ void erf_parts(float g, float& erfv, float& gauss) {
  const float x = fabsf(g) * 0.70710678118654752f;
  const float t = __fdividef(1.f, fmaf(0.3275911f, x, 1.f));
  gauss = __expf(-x * x);
  float p = fmaf(t, 1.061405429f, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  erfv = copysignf(1.f - p * t * gauss, g);
}
__device__ __forceinline__ float gelu_erf(float g) {
  float e, ex;
  erf_parts(g, e, ex);
  return 0.5f * g * (1.f + e);
}
// gelu(g) and d gelu / dg from one evaluation
__device__ __forceinline__ void gelu_erf_both(float g, float& y, float& dy) {
  float e, ex;
  erf_parts(g, e, ex);
  const float cdf = 0.5f * (1.f + e);
  y = g * cdf;
  dy = fmaf(g * 0.3989422804014327f, ex, cdf);
}

__global__ void geglu_fwd_kernel(const bf16* __restrict__ u, bf16* __restrict__ y, long long M, int F) {
  const int nv = F >> 3;
  const long long total = M * nv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / nv;
    const int v = (int)(i % nv);
    float a[8], g[8];
    load8(u + r * 2 * F + v * 8, a);
    load8(u + r * 2 * F + F + v * 8, g);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] *= gelu_erf(g[j]);
    store8(y + r * F + v * 8, a);
  }
}

__global__ void geglu_bwd_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ u, bf16* __restrict__ du, long long M, int F) {
  const int nv = F >> 3;
  const long long total = M * nv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / nv;
    const int v = (int)(i % nv);
    float a[8], g[8], d[8], da[8], dg[8];
    load8(u + r * 2 * F + v * 8, a);
    load8(u + r * 2 * F + F + v * 8, g);
    load8(dy + r * F + v * 8, d);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float ge, gd;
      gelu_erf_both(g[j], ge, gd);
      da[j] = d[j] * ge;
      dg[j] = d[j] * a[j] * gd;
    }
    store8(du + r * 2 * F + v * 8, da);
    store8(du + r * 2 * F + F + v * 8, dg);
  }
}

// ------------------------------------------------------------------------------------------------ misc elementwise
__global__ void add_bf16_kernel(const bf16* __restrict__ a, const bf16* __restrict__ b, bf16* __restrict__ y, long long nvec) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    float fa[8], fb[8];
    load8(a + i * 8, fa);
    load8(b + i * 8, fb);
#pragma unroll
    for (int j = 0; j < 8; ++j) fa[j] += fb[j];
    store8(y + i * 8, fa);
  }
}

__global__ void silu_f32_to_bf16_kernel(const float* __restrict__ x, bf16* __restrict__ y, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    y[i] = __float2bfloat16(silu_f(x[i]));
}
__global__ void silu_bwd_f32_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dx[i] = dy[i] * silu_grad_f(x[i]);
}

__global__ void copy2d_kernel(const bf16* __restrict__ src, long long ld_src, bf16* __restrict__ dst, long long ld_dst, long long rows, int nvec) {
  const long long total = rows * nvec;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / nvec;
    const int v = (int)(i % nvec);
    st16(dst + r * ld_dst + v * 8, ld16(src + r * ld_src + v * 8));
  }
}

__global__ void upsample2_fwd_kernel(const bf16* __restrict__ x, bf16* __restrict__ y, long long rows_in, int L, int nvec) {
  const long long total = rows_in * nvec;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / nvec;  // b*L + l
    const int v = (int)(i % nvec);
    const bf16x8 t = ld16(x + (r * nvec + v) * 8);
    st16(y + ((2 * r) * nvec + v) * 8, t);
    st16(y + ((2 * r + 1) * nvec + v) * 8, t);
  }
}
__global__ void upsample2_bwd_kernel(const bf16* __restrict__ dy, bf16* __restrict__ dx, long long rows_in, int nvec) {
  const long long total = rows_in * nvec;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / nvec;
    const int v = (int)(i % nvec);
    float a[8], b[8];
    load8(dy + ((2 * r) * nvec + v) * 8, a);
    load8(dy + ((2 * r + 1) * nvec + v) * 8, b);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] += b[j];
    store8(dx + (r * nvec + v) * 8, a);
  }
}

// [B, C, L] fp32 <-> [B, L, C] bf16 through a 32x32 shared tile (both sides coalesced)
__global__ void ncl_to_nlc_kernel(const float* __restrict__ x, bf16* __restrict__ y, int C, int L) {
  __shared__ float t[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, l0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, l = l0 + threadIdx.x;
    if (c < C && l < L) t[i][threadIdx.x] = x[((long long)b * C + c) * L + l];
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int l = l0 + i, c = c0 + threadIdx.x;
    if (c < C && l < L) y[((long long)b * L + l) * C + c] = __float2bfloat16(t[threadIdx.x][i]);
  }
}
__global__ void nlc_to_ncl_kernel(const bf16* __restrict__ x, float* __restrict__ y, int C, int L) {
  __shared__ float t[32][33];
  const int b = blockIdx.z, c0 = blockIdx.y * 32, l0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int l = l0 + i, c = c0 + threadIdx.x;
    if (c < C && l < L) t[i][threadIdx.x] = __bfloat162float(x[((long long)b * L + l) * C + c]);
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, l = l0 + threadIdx.x;
    if (c < C && l < L) y[((long long)b * C + c) * L + l] = t[threadIdx.x][i];
  }
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ x, bf16* __restrict__ y, long long n) {
  const long long nv = n >> 3;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
    const float4 a = *reinterpret_cast<const float4*>(x + i * 8), b = *reinterpret_cast<const float4*>(x + i * 8 + 4);
    float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    store8(y + i * 8, f);
  }
  if (blockIdx.x == 0)
    for (long long i = nv * 8 + threadIdx.x; i < n; i += blockDim.x) y[i] = __float2bfloat16(x[i]);
}
__global__ void cast_bf16_f32_kernel(const bf16* __restrict__ x, float* __restrict__ y, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) y[i] = __bfloat162float(x[i]);
}

// [Co, Ci, k] fp32 -> [Co, k*Ci] bf16 (tap-major K axis so that each tap is a contiguous K segment)
__global__ void pack_conv_weight_kernel(const float* __restrict__ w, bf16* __restrict__ wp, long long Co, int Ci, int k) {
  const long long total = Co * Ci * k;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long co = i / ((long long)Ci * k);
    const int rem = (int)(i % ((long long)Ci * k));
    const int t = rem / Ci, ci = rem % Ci;  // destination order
    wp[i] = __float2bfloat16(w[(co * Ci + ci) * k + t]);
  }
}
__global__ void unpack_conv_wgrad_kernel(const float* __restrict__ gp, float* __restrict__ g, long long Co, int Ci, int k, int accumulate) {
  const long long total = Co * Ci * k;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long co = i / ((long long)Ci * k);
    const int rem = (int)(i % ((long long)Ci * k));
    const int ci = rem / k, t = rem % k;  // destination order [Co, Ci, k]
    const float v = gp[(co * k + t) * Ci + ci];
    g[i] = accumulate ? g[i] + v : v;
  }
}

// out[c] += sum_r x[r, c].  grid = (column blocks of 256, row chunks, batch).  A warp reads 32 consecutive 16-byte
// vectors of one row (512 contiguous bytes); the 8 warps of a CTA take rows w, w+8, ... four at a time (four independent
// loads in flight per thread); partials are combined through shared memory and leave as one atomicAdd per (CTA, column).
__global__ void __launch_bounds__(256) colsum_kernel(const bf16* __restrict__ x, long long ld, float* __restrict__ out, long long rows, int cols,
                                                     int rows_per_cta, long long batch_stride, long long out_stride) {
  __shared__ float sh[8][256];
  x += (long long)blockIdx.z * batch_stride;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 256 + lane * 8;
  const long long r0 = (long long)blockIdx.y * rows_per_cta;
  const long long r1 = min(rows, r0 + rows_per_cta);
  float s[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = 0.f;
  if (c < cols) {
    const bf16* xc = x + c;
    long long r = r0 + warp;
    for (; r + 24 < r1; r += 32) {
      float f0[8], f1[8], f2[8], f3[8];
      load8(xc + r * ld, f0);
      load8(xc + (r + 8) * ld, f1);
      load8(xc + (r + 16) * ld, f2);
      load8(xc + (r + 24) * ld, f3);
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += (f0[j] + f1[j]) + (f2[j] + f3[j]);
    }
    for (; r < r1; r += 8) {
      float f0[8];
      load8(xc + r * ld, f0);
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += f0[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) sh[warp][lane * 8 + j] = s[j];
  __syncthreads();
  const int cc = blockIdx.x * 256 + threadIdx.x;
  if (cc < cols) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += sh[w][threadIdx.x];
    atomicAdd(&out[(long long)blockIdx.z * out_stride + cc], t);
  }
}

// The same reduction sized to run BESIDE a persistent GEMM / attention CTA on the same SM (those leave ~11 K registers and ~8 KB of
// shared memory per SM): 128 threads, 4 KB of shared memory.  Bias gradients are off the backward's critical path; launched on a
// second stream they fill the SMs' idle resources and the gaps at kernel boundaries instead of a slot of their own in the stream.
__global__ void __launch_bounds__(128, 4) colsum_lite_kernel(const bf16* __restrict__ x, long long ld, float* __restrict__ out, long long rows, int cols,
                                                             int rows_per_cta, long long batch_stride, long long out_stride) {
  __shared__ float sh[4][256];
  x += (long long)blockIdx.z * batch_stride;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 256 + lane * 8;
  const long long r0 = (long long)blockIdx.y * rows_per_cta;
  const long long r1 = min(rows, r0 + rows_per_cta);
  float s[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = 0.f;
  if (c < cols) {
    const bf16* xc = x + c;
    long long r = r0 + warp;
    for (; r + 12 < r1; r += 16) {
      float f0[8], f1[8], f2[8], f3[8];
      load8(xc + r * ld, f0);
      load8(xc + (r + 4) * ld, f1);
      load8(xc + (r + 8) * ld, f2);
      load8(xc + (r + 12) * ld, f3);
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += (f0[j] + f1[j]) + (f2[j] + f3[j]);
    }
    for (; r < r1; r += 4) {
      float f0[8];
      load8(xc + r * ld, f0);
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += f0[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) sh[warp][lane * 8 + j] = s[j];
  __syncthreads();
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int cl = threadIdx.x + h * 128;
    const int cc = blockIdx.x * 256 + cl;
    if (cc < cols) atomicAdd(&out[(long long)blockIdx.z * out_stride + cc], (sh[0][cl] + sh[1][cl]) + (sh[2][cl] + sh[3][cl]));
  }
}

__global__ void time_sinusoid_kernel(const int64_t* __restrict__ t, float* __restrict__ out, int B, int dim) {
  const int half = dim / 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * half) return;
  const int b = i / half, k = i % half;
  const float freq = expf(-9.210340371976184f * (float)k / (float)half);  // ln(10000)
  const float ang = (float)t[b] * freq;
  out[(long long)b * dim + k] = cosf(ang);          // flip_sin_to_cos=True: [cos | sin]
  out[(long long)b * dim + half + k] = sinf(ang);
}

__global__ void text_embed_fwd_kernel(const int32_t* __restrict__ ids, const float* __restrict__ E, const float* __restrict__ pe,
                                      bf16* __restrict__ y, long long BL, int L, int D, int V) {
  const int nv = D >> 3;
  const long long total = BL * nv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / nv;
    const int v = (int)(i % nv);
    const int l = (int)(r % L);
    const int id = min(max(ids[r], 0), V - 1);     // nn.Embedding raises on an out-of-range id; a kernel cannot, so it never reads outside E
    const float* e = E + (long long)id * D + v * 8;
    const float* p = pe + (long long)l * D + v * 8;
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = e[j] + p[j];
    store8(y + r * D + v * 8, f);
  }
}
// dE[v, :] += sum over positions p with ids[p] == v of dy[p, :].  The vocabulary is tiny (150 rows) and the padding id takes ~40 % of
// the positions, so scattering with atomics serialises on a handful of addresses.  Instead: CTA (v, chunk) scans its chunk of the
// ids, gathers the matching rows into registers (thread t owns 16-byte vectors t, t + blockDim, ...) and flushes once.
constexpr int EMB_MAXV = 4;      // vectors per thread: D <= 8 * EMB_MAXV * 256
__global__ void __launch_bounds__(256) text_embed_bwd_kernel(const int32_t* __restrict__ ids, const bf16* __restrict__ dy, float* __restrict__ dE,
                                                             long long BL, int D, int per_chunk) {
  const int v = blockIdx.x;
  const long long p0 = (long long)blockIdx.y * per_chunk, p1 = min(BL, p0 + per_chunk);
  const int nv = D >> 3;
  float acc[EMB_MAXV][8];
#pragma unroll
  for (int k = 0; k < EMB_MAXV; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[k][j] = 0.f;
  __shared__ int hits[256];
  __shared__ int nhit;
  bool any = false;
  for (long long base = p0; base < p1; base += blockDim.x) {
    if (threadIdx.x == 0) nhit = 0;
    __syncthreads();
    const long long pp = base + threadIdx.x;
    if (pp < p1 && ids[pp] == v) hits[atomicAdd(&nhit, 1)] = (int)(pp - base);   // order within a batch of 256 positions does not matter
    __syncthreads();
    const int n = nhit;
    for (int hh = 0; hh < n; hh += 4) {       // four independent row gathers in flight
      const bf16* row[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) row[u] = dy + (base + hits[min(hh + u, n - 1)]) * D;
#pragma unroll
      for (int k = 0; k < EMB_MAXV; ++k) {
        const int vec = threadIdx.x + k * blockDim.x;
        if (vec < nv) {
          float f[4][8];
#pragma unroll
          for (int u = 0; u < 4; ++u) load8(row[u] + vec * 8, f[u]);
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (hh + u < n) {
#pragma unroll
              for (int j = 0; j < 8; ++j) acc[k][j] += f[u][j];
            }
        }
      }
    }
    any |= n > 0;
    __syncthreads();
  }
  if (!any) return;
#pragma unroll
  for (int k = 0; k < EMB_MAXV; ++k) {
    const int vec = threadIdx.x + k * blockDim.x;
    if (vec < nv) {
      float* d = dE + (long long)v * D + vec * 8;
#pragma unroll
      for (int j = 0; j < 8; ++j) atomicAdd(d + j, acc[k][j]);
    }
  }
}

}  // namespace

#define ST ((cudaStream_t)stream)

extern "C" int pt_softmax_fwd(const float* S, void* P, int64_t rows, int n, int64_t ld_s, int64_t ld_p, void* stream) {
  PT_REQUIRE(rows > 0 && n > 0 && n <= SM_MAXV * 128 && ld_s % 4 == 0 && ld_p % 4 == 0 && ld_s >= (n + 3) / 4 * 4 && ld_p >= (n + 3) / 4 * 4,
             "softmax_fwd: rows=%lld n=%d ld_s=%lld ld_p=%lld", (long long)rows, n, (long long)ld_s, (long long)ld_p);
  softmax_fwd_kernel<<<grid_for(rows, 8), 256, 0, ST>>>(S, (bf16*)P, rows, n, ld_s, ld_p);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_softmax_bwd(const float* dP, const void* P, void* dS, int64_t rows, int n, int64_t ld_s, int64_t ld_p, float scale,
                              void* stream) {
  PT_REQUIRE(rows > 0 && n > 0 && n <= SM_MAXV * 128 && ld_s % 4 == 0 && ld_p % 4 == 0 && ld_s >= (n + 3) / 4 * 4 && ld_p >= (n + 3) / 4 * 4,
             "softmax_bwd: rows=%lld n=%d", (long long)rows, n);
  softmax_bwd_kernel<<<grid_for(rows, 8), 256, 0, ST>>>(dP, (const bf16*)P, (bf16*)dS, rows, n, ld_s, ld_p, scale);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_geglu_fwd(const void* u, void* y, int64_t M, int F, void* stream) {
  PT_REQUIRE(M > 0 && F > 0 && F % 8 == 0, "geglu_fwd: M=%lld F=%d", (long long)M, F);
  geglu_fwd_kernel<<<grid_for(M * (F / 8), 256), 256, 0, ST>>>((const bf16*)u, (bf16*)y, M, F);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_geglu_bwd(const void* dy, const void* u, void* du, int64_t M, int F, void* stream) {
  PT_REQUIRE(M > 0 && F > 0 && F % 8 == 0, "geglu_bwd: M=%lld F=%d", (long long)M, F);
  geglu_bwd_kernel<<<grid_for(M * (F / 8), 256), 256, 0, ST>>>((const bf16*)dy, (const bf16*)u, (bf16*)du, M, F);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_add_bf16(const void* a, const void* b, void* y, int64_t n, void* stream) {
  PT_REQUIRE(n > 0 && n % 8 == 0, "add_bf16: n=%lld must be a multiple of 8", (long long)n);
  add_bf16_kernel<<<grid_for(n / 8, 256), 256, 0, ST>>>((const bf16*)a, (const bf16*)b, (bf16*)y, n / 8);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_silu_f32_to_bf16(const float* x, void* y, int64_t n, void* stream) {
  PT_REQUIRE(n > 0, "silu: n=%lld", (long long)n);
  silu_f32_to_bf16_kernel<<<grid_for(n, 256), 256, 0, ST>>>(x, (bf16*)y, n);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_silu_bwd_f32(const float* x, const float* dy, float* dx, int64_t n, void* stream) {
  PT_REQUIRE(n > 0, "silu_bwd: n=%lld", (long long)n);
  silu_bwd_f32_kernel<<<grid_for(n, 256), 256, 0, ST>>>(x, dy, dx, n);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_copy2d_bf16(const void* src, int64_t ld_src, void* dst, int64_t ld_dst, int64_t rows, int cols, void* stream) {
  PT_REQUIRE(rows > 0 && cols > 0 && cols % 8 == 0 && ld_src % 8 == 0 && ld_dst % 8 == 0, "copy2d: rows=%lld cols=%d", (long long)rows, cols);
  copy2d_kernel<<<grid_for(rows * (cols / 8), 256), 256, 0, ST>>>((const bf16*)src, ld_src, (bf16*)dst, ld_dst, rows, cols / 8);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_upsample2_fwd(const void* x, void* y, int B, int L, int C, void* stream) {
  PT_REQUIRE(B > 0 && L > 0 && C % 8 == 0, "upsample2_fwd: C=%d", C);
  upsample2_fwd_kernel<<<grid_for((long long)B * L * (C / 8), 256), 256, 0, ST>>>((const bf16*)x, (bf16*)y, (long long)B * L, L, C / 8);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_upsample2_bwd(const void* dy, void* dx, int B, int L, int C, void* stream) {
  PT_REQUIRE(B > 0 && L > 0 && C % 8 == 0, "upsample2_bwd: C=%d", C);
  upsample2_bwd_kernel<<<grid_for((long long)B * L * (C / 8), 256), 256, 0, ST>>>((const bf16*)dy, (bf16*)dx, (long long)B * L, C / 8);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_ncl_f32_to_nlc_bf16(const float* x, void* y, int B, int C, int L, void* stream) {
  PT_REQUIRE(B > 0 && C > 0 && L > 0 && B <= 65535, "ncl_to_nlc: B=%d C=%d L=%d", B, C, L);
  ncl_to_nlc_kernel<<<dim3((L + 31) / 32, (C + 31) / 32, B), dim3(32, 8), 0, ST>>>(x, (bf16*)y, C, L);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_nlc_bf16_to_ncl_f32(const void* x, float* y, int B, int C, int L, void* stream) {
  PT_REQUIRE(B > 0 && C > 0 && L > 0 && B <= 65535, "nlc_to_ncl: B=%d C=%d L=%d", B, C, L);
  nlc_to_ncl_kernel<<<dim3((L + 31) / 32, (C + 31) / 32, B), dim3(32, 8), 0, ST>>>((const bf16*)x, y, C, L);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_cast_f32_to_bf16(const float* x, void* y, int64_t n, void* stream) {
  PT_REQUIRE(n > 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0, "cast: n=%lld / alignment", (long long)n);
  cast_f32_bf16_kernel<<<grid_for(n / 8 + 1, 256), 256, 0, ST>>>(x, (bf16*)y, n);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_cast_bf16_to_f32(const void* x, float* y, int64_t n, void* stream) {
  PT_REQUIRE(n > 0, "cast: n=%lld", (long long)n);
  cast_bf16_f32_kernel<<<grid_for(n, 256), 256, 0, ST>>>((const bf16*)x, y, n);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_pack_conv_weight(const float* w, void* wp, int Co, int Ci, int k, void* stream) {
  PT_REQUIRE(Co > 0 && Ci > 0 && k > 0, "pack_conv_weight: Co=%d Ci=%d k=%d", Co, Ci, k);
  pack_conv_weight_kernel<<<grid_for((long long)Co * Ci * k, 256), 256, 0, ST>>>(w, (bf16*)wp, Co, Ci, k);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_unpack_conv_wgrad(const float* gp, float* g, int Co, int Ci, int k, int accumulate, void* stream) {
  PT_REQUIRE(Co > 0 && Ci > 0 && k > 0, "unpack_conv_wgrad: Co=%d Ci=%d k=%d", Co, Ci, k);
  unpack_conv_wgrad_kernel<<<grid_for((long long)Co * Ci * k, 256), 256, 0, ST>>>(gp, g, Co, Ci, k, accumulate);
  PT_LAUNCH_CHECK();
  return PT_OK;
}

static int colsum_launch(const bf16* x, long long ld, float* out, long long rows, int cols, int nbatch, long long batch_stride,
                         long long out_stride, cudaStream_t st, bool lite = false) {
  PT_REQUIRE(cols % 8 == 0 && ld % 8 == 0 && nbatch >= 1 && nbatch <= 65535, "colsum: cols=%d", cols);
  const int cblocks = (cols + 255) / 256;
  long long want = (8ll * pt_num_sms() + (long long)nbatch * cblocks - 1) / ((long long)nbatch * cblocks);
  if (want < 1) want = 1;
  long long rpc = (rows + want - 1) / want;
  if (rpc < 64) rpc = 64;
  const unsigned rchunks = (unsigned)((rows + rpc - 1) / rpc);
  PT_REQUIRE(rchunks <= 65535, "colsum: too many row chunks");
  if (lite)
    colsum_lite_kernel<<<dim3(cblocks, rchunks, nbatch), 128, 0, st>>>(x, ld, out, rows, cols, (int)rpc, batch_stride, out_stride);
  else
    colsum_kernel<<<dim3(cblocks, rchunks, nbatch), 256, 0, st>>>(x, ld, out, rows, cols, (int)rpc, batch_stride, out_stride);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_colsum_bf16(const void* x, int64_t ld, float* out, int64_t rows, int cols, void* stream) {
  PT_REQUIRE(rows > 0 && cols > 0, "colsum: rows=%lld cols=%d", (long long)rows, cols);
  return colsum_launch((const bf16*)x, ld, out, rows, cols, 1, 0, cols, ST);
}
extern "C" int pt_colsum_bf16_lite(const void* x, int64_t ld, float* out, int64_t rows, int cols, void* stream) {
  PT_REQUIRE(rows > 0 && cols > 0, "colsum: rows=%lld cols=%d", (long long)rows, cols);
  return colsum_launch((const bf16*)x, ld, out, rows, cols, 1, 0, cols, ST, true);
}
extern "C" int pt_batch_colsum_bf16(const void* x, float* out, int64_t out_stride, int B, int L, int C, void* stream) {
  PT_REQUIRE(B > 0 && L > 0 && C > 0 && out_stride >= C, "batch_colsum: B=%d L=%d C=%d", B, L, C);
  PT_CUDA_OK(cudaMemset2DAsync(out, sizeof(float) * out_stride, 0, sizeof(float) * C, B, ST));
  return colsum_launch((const bf16*)x, C, out, L, C, B, (long long)L * C, out_stride, ST);
}
extern "C" int pt_time_sinusoid(const int64_t* t, float* out, int B, int dim, void* stream) {
  PT_REQUIRE(B > 0 && dim > 0 && dim % 2 == 0, "time_sinusoid: B=%d dim=%d", B, dim);
  time_sinusoid_kernel<<<(B * dim / 2 + 127) / 128, 128, 0, ST>>>(t, out, B, dim);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_text_embed_fwd(const int32_t* ids, const float* E, const float* pe, void* y, int B, int L, int D, int V, void* stream) {
  PT_REQUIRE(B > 0 && L > 0 && D % 8 == 0 && V > 0, "text_embed_fwd: D=%d", D);
  text_embed_fwd_kernel<<<grid_for((long long)B * L * (D / 8), 256), 256, 0, ST>>>(ids, E, pe, (bf16*)y, (long long)B * L, L, D, V);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
extern "C" int pt_text_embed_bwd(const int32_t* ids, const void* dy, float* dE, int B, int L, int D, int V, void* stream) {
  PT_REQUIRE(B > 0 && L > 0 && D % 8 == 0 && V > 0, "text_embed_bwd: D=%d", D);
  PT_REQUIRE(D <= 8 * EMB_MAXV * 256 && V <= 65535, "text_embed_bwd: D=%d V=%d", D, V);
  const long long BL = (long long)B * L;
  int chunks = (int)((BL + 511) / 512);              // ~512 positions per CTA: the padding id's rows are spread over many CTAs
  if (chunks > 256) chunks = 256;
  const int per_chunk = (int)((BL + chunks - 1) / chunks);
  const int threads = (D / 8) >= 256 ? 256 : (((D / 8) + 31) / 32 * 32);
  text_embed_bwd_kernel<<<dim3(V, chunks), threads, 0, ST>>>(ids, (const bf16*)dy, dE, BL, D, per_chunk);
  PT_LAUNCH_CHECK();
  return PT_OK;
}
