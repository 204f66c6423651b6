// e4t_b200 — HBM-bound normalisation kernels on NHWC / token-major bf16 activations (fp32 statistics).
//   GroupNorm(32)+SiLU : diffusers ResnetBlock2D.norm1/norm2, Transformer2DModel.norm (transformer_2d.py:149,253),
//                        UNet conv_norm_out (unet_2d_condition.py:554-556)
//   LayerNorm          : BasicTransformerBlock.norm1/2/3 (attention.py:258-273)
// Coalesced 16-byte / 4-byte vector loads, warp-shuffle + shared-memory reductions, grids sized well past 148 SMs.
#include "common.cuh"
#include <stdlib.h>

// ---------------------------------------------------------------------------------------------
// GroupNorm statistics: sums[b][g] = (sum x, sum x^2) over HW x (C/G) elements.   (sums pre-zeroed)
// mode 0: plain stats of x.
// mode 1: backward stats: (sum dxhat, sum dxhat*xhat) with dxhat = dy * act'(y0) * gamma.
// ---------------------------------------------------------------------------------------------
// Thread mapping (all four kernels): a thread owns ONE 8-channel vector column (16-byte loads, coalesced across
// the warp) and walks rows; its per-channel constants live in registers.  blockDim = vpr * k (vpr = C/8 vector
// columns, k = rows handled concurrently by one CTA), so no thread is idle and no per-element smem lookups occur.
static constexpr int kGNMaxThreads = 320;

struct GNChan {
  float mean, rstd, gamma, beta;
};

// sigmoid through ONE MUFU operation (tanh.approx, |err| ~ 2^-11): the exp + reciprocal form costs two, and the
// GroupNorm+SiLU apply pass was 47 % MUFU-busy (ncu r02) on top of its memory traffic
__device__ __forceinline__ float sigmoid_fast(float y) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * y));
  return fmaf(0.5f, t, 0.5f);
}
__device__ __forceinline__ float silu_fast(float y) { return y * sigmoid_fast(y); }
__device__ __forceinline__ float silu_grad(float y) {
  const float sg = sigmoid_fast(y);
  return sg * (1.f + y * (1.f - sg));
}
__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
  const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  return make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
}
// The forward sums of group g of image b are taken about a pivot, the group's first element p = x[b][0][g * cpg]:
// (Σ(x - p), Σ(x - p)²).  Σx² / n - mean² would lose the variance to cancellation, with a relative error that grows as
// (mean / std)²; about a sample of the group the two terms are of the order of the variance itself.
__device__ __forceinline__ float gn_pivot(const bf16* __restrict__ x, int b, int g, int HW, int C, int cpg) {
  return __bfloat162float(x[(long)b * HW * C + g * cpg]);
}
__device__ __forceinline__ void gn_mean_rstd(const float* __restrict__ stats, const bf16* __restrict__ x, int b, int g,
                                             int HW, int C, int G, float inv_n, float eps, float& mean, float& rstd) {
  const float d = stats[((long)b * G + g) * 2] * inv_n, ss = stats[((long)b * G + g) * 2 + 1] * inv_n;
  mean = gn_pivot(x, b, g, HW, C, C / G) + d;
  rstd = rsqrtf(fmaxf(ss - d * d, 0.f) + eps);
}
// per-channel (mean, rstd, gamma, beta) of this thread's 8 channels, from the forward sums
__device__ __forceinline__ void gn_thread_chan(GNChan* ch, const float* __restrict__ stats, const bf16* __restrict__ x,
                                               const float* __restrict__ gamma, const float* __restrict__ beta, int b,
                                               int c0, int HW, int C, int G, float inv_n, float eps) {
  const int cpg = C / G;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    gn_mean_rstd(stats, x, b, (c0 + j) / cpg, HW, C, G, inv_n, eps, ch[j].mean, ch[j].rstd);
    ch[j].gamma = gamma[c0 + j];
    ch[j].beta = beta[c0 + j];
  }
}

// sums[b][g] += (Σ a, Σ b) over this CTA's rows.  MODE 0: (x - p, (x - p)²), p = the group's pivot (gn_pivot).
// MODE 1: (dxhat, dxhat·xhat).
template <int MODE>
__global__ void __launch_bounds__(kGNMaxThreads)
gn_stats_kernel(const bf16* __restrict__ x, const bf16* __restrict__ dy, const float* __restrict__ fstats,
                const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ sums, int HW,
                int C, int G, int rows_per_cta, float eps, int act) {
  extern __shared__ __align__(16) uint8_t gsm[];
  float2* schan = reinterpret_cast<float2*>(gsm);  // [rstep][C] per-(row-lane, channel) partials
  const int b = blockIdx.y;
  const int vpr = C / 8;
  const int cv = threadIdx.x % vpr, rl = threadIdx.x / vpr, rstep = blockDim.x / vpr;
  const int c0 = cv * 8;
  const int r0 = blockIdx.x * rows_per_cta;
  const int r1 = min(HW, r0 + rows_per_cta);
  GNChan ch[8];
  float piv[8];
  if (MODE == 1) gn_thread_chan(ch, fstats, x, gamma, beta, b, c0, HW, C, G, 1.f / ((float)HW * (float)(C / G)), eps);
  __syncthreads();
  float a0[8], a1[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    a0[j] = a1[j] = 0.f;
    if (MODE == 0) piv[j] = gn_pivot(x, b, (c0 + j) / (C / G), HW, C, C / G);
  }
  const bf16* xb = x + ((long)b * HW) * C + c0;
  const bf16* db = MODE == 1 ? dy + ((long)b * HW) * C + c0 : nullptr;
#pragma unroll 4
  for (int r = r0 + rl; r < r1; r += rstep) {
    float xv[8];
    unpack8(*reinterpret_cast<const uint4*>(xb + (long)r * C), xv);
    if (MODE == 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float d = xv[j] - piv[j];
        a0[j] += d;
        a1[j] += d * d;
      }
    } else {
      float dv[8];
      unpack8(*reinterpret_cast<const uint4*>(db + (long)r * C), dv);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float xh = (xv[j] - ch[j].mean) * ch[j].rstd;
        float g = dv[j] * ch[j].gamma;
        if (act) g *= silu_grad(xh * ch[j].gamma + ch[j].beta);
        a0[j] += g;
        a1[j] += g * xh;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) schan[rl * C + c0 + j] = make_float2(a0[j], a1[j]);
  __syncthreads();
  const int cpg = C / G;
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    float s = 0.f, ss = 0.f;
    for (int q = 0; q < rstep; ++q)
      for (int i = 0; i < cpg; ++i) {
        const float2 p = schan[q * C + g * cpg + i];
        s += p.x;
        ss += p.y;
      }
    atomicAdd(&sums[((long)b * G + g) * 2], s);
    atomicAdd(&sums[((long)b * G + g) * 2 + 1], ss);
  }
}

// MODE 0: y = act(xhat*gamma+beta).   MODE 1: dx = rstd*(dxhat - mean(dxhat) - xhat*mean(dxhat*xhat)).
template <int MODE>
__global__ void __launch_bounds__(kGNMaxThreads)
gn_apply_kernel(const bf16* __restrict__ x, const bf16* __restrict__ dy, const float* __restrict__ fstats,
                const float* __restrict__ bstats, const float* __restrict__ gamma, const float* __restrict__ beta,
                bf16* __restrict__ out, int HW, int C, int G, int rows_per_cta, float eps, int act) {
  const int b = blockIdx.y;
  const float inv_n = 1.f / ((float)HW * (float)(C / G));
  const int vpr = C / 8;
  const int cv = threadIdx.x % vpr, rl = threadIdx.x / vpr, rstep = blockDim.x / vpr;
  const int c0 = cv * 8;
  GNChan ch[8];
  gn_thread_chan(ch, fstats, x, gamma, beta, b, c0, HW, C, G, inv_n, eps);
  float scale[8], shift[8], m1[8], m2[8];
  const int cpg = C / G;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    scale[j] = ch[j].rstd * ch[j].gamma;
    shift[j] = ch[j].beta - ch[j].mean * scale[j];
    if (MODE == 1) {
      const int g = (c0 + j) / cpg;
      m1[j] = bstats[((long)b * G + g) * 2] * inv_n;
      m2[j] = bstats[((long)b * G + g) * 2 + 1] * inv_n;
    }
  }
  const int r0 = blockIdx.x * rows_per_cta;
  const int r1 = min(HW, r0 + rows_per_cta);
  const long base = ((long)b * HW) * C + c0;
#pragma unroll 4
  for (int r = r0 + rl; r < r1; r += rstep) {
    float xv[8], o[8];
    unpack8(*reinterpret_cast<const uint4*>(x + base + (long)r * C), xv);
    if (MODE == 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        o[j] = fmaf(xv[j], scale[j], shift[j]);
        if (act) o[j] = silu_fast(o[j]);
      }
    } else {
      float dv[8];
      unpack8(*reinterpret_cast<const uint4*>(dy + base + (long)r * C), dv);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float xh = (xv[j] - ch[j].mean) * ch[j].rstd;
        float g = dv[j] * ch[j].gamma;
        if (act) g *= silu_grad(fmaf(xv[j], scale[j], shift[j]));
        o[j] = ch[j].rstd * (g - m1[j] - xh * m2[j]);
      }
    }
    *reinterpret_cast<uint4*>(out + base + (long)r * C) = pack8(o);
  }
}

// Tuning overrides (unset = the heuristics below): E4T_GN_ROWS = rows per CTA, E4T_GN_THREADS = target block size.
static int gn_env(const char* name) {
  const char* e = getenv(name);
  return e ? atoi(e) : 0;
}
// rows per CTA such that the grid is (about) ONE full wave of resident CTAs: the round-1 choice (64 rows, >= 8 CTAs per
// SM "overall") gave 1.73 waves at the 16 x 1024 x 1280 shape, i.e. a second wave that is three-quarters empty
template <typename K>
static int gn_rows_per_cta(K kernel, int threads, size_t smem_per_rl, int C, int B, int HW) {
  const int forced = gn_env("E4T_GN_ROWS");
  if (forced > 0) return forced;
  int occ = 0;
  const size_t smem = smem_per_rl * (size_t)(threads / (C / 8));
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem) != cudaSuccess || occ < 1) occ = 4;
  int sms = 0, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (sms <= 0) sms = 148;
  const long target = (long)sms * occ;
  long chunks = target / B;                 // row chunks per image
  if (chunks < 1) chunks = 1;
  if (chunks > HW) chunks = HW;
  int rows = cdiv(HW, chunks);
  const int rstep = threads / (C / 8);
  if (rows < rstep) rows = rstep;           // at least one row per concurrent row lane
  return rows;
}
static int gn_block(int C) {
  const int vpr = C / 8;
  int target = gn_env("E4T_GN_THREADS");
  if (target <= 0 || target > kGNMaxThreads) target = 256;
  int k = target / vpr;
  if (k < 1) k = 1;
  return vpr * k;
}

// stats: fp32 [B][G][2] = (Σ(x - p), Σ(x - p)²) about the pivot p = x[b][0][g * C / G]; written by this call.
extern "C" int e4t_groupnorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* stats, int B,
                                 int HW, int C, int G, float eps, int act_silu, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  E4T_CHECK(C % G == 0 && C % 8 == 0 && C / 8 <= kGNMaxThreads, "e4t_groupnorm_fwd: unsupported C=%d G=%d", C, G);
  E4T_CUDA(cudaMemsetAsync(stats, 0, (size_t)B * G * 2 * sizeof(float), st));
  const int threads = gn_block(C);
  const int rows = gn_rows_per_cta(gn_stats_kernel<0>, threads, (size_t)C * sizeof(float2), C, B, HW);
  dim3 grid(cdiv(HW, rows), B);
  gn_stats_kernel<0><<<grid, threads, (size_t)(threads / (C / 8)) * C * sizeof(float2), st>>>((const bf16*)x, nullptr, nullptr, nullptr,
                                                                        nullptr, stats, HW, C, G, rows, eps, 0);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  const int rows_a = gn_rows_per_cta(gn_apply_kernel<0>, threads, 0, C, B, HW);
  gn_apply_kernel<0><<<dim3(cdiv(HW, rows_a), B), threads, 0, st>>>((const bf16*)x, nullptr, stats, nullptr, gamma, beta,
                                                                    (bf16*)y, HW, C, G, rows_a, eps, act_silu);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// dx only (gamma/beta are frozen on the pre-training path).  scratch: fp32 [B][G][2].
extern "C" int e4t_groupnorm_bwd(const void* x, const void* dy, const float* gamma, const float* beta,
                                 const float* stats, void* dx, float* scratch, int B, int HW, int C, int G, float eps,
                                 int act_silu, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  E4T_CHECK(C % G == 0 && C % 8 == 0 && C / 8 <= kGNMaxThreads, "e4t_groupnorm_bwd: unsupported C=%d G=%d", C, G);
  E4T_CUDA(cudaMemsetAsync(scratch, 0, (size_t)B * G * 2 * sizeof(float), st));
  const int threads = gn_block(C);
  const int rows = gn_rows_per_cta(gn_stats_kernel<1>, threads, (size_t)C * sizeof(float2), C, B, HW);
  dim3 grid(cdiv(HW, rows), B);
  gn_stats_kernel<1><<<grid, threads, (size_t)(threads / (C / 8)) * C * sizeof(float2), st>>>((const bf16*)x, (const bf16*)dy, stats, gamma,
                                                                        beta, scratch, HW, C, G, rows, eps, act_silu);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  const int rows_a = gn_rows_per_cta(gn_apply_kernel<1>, threads, 0, C, B, HW);
  gn_apply_kernel<1><<<dim3(cdiv(HW, rows_a), B), threads, 0, st>>>((const bf16*)x, (const bf16*)dy, stats, scratch, gamma,
                                                                    beta, (bf16*)dx, HW, C, G, rows_a, eps, act_silu);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// LayerNorm over the last dim (C <= 2048, C % 8 == 0): one warp per row, values held in registers.
// ---------------------------------------------------------------------------------------------
template <int MODE, int kLNMaxIter>  // MODE 0 fwd, 1 bwd(dx); kLNMaxIter = ceil(C / 256)
__global__ void __launch_bounds__(256)
ln_kernel(const bf16* __restrict__ x, const bf16* __restrict__ dy, const float* __restrict__ gamma,
          const float* __restrict__ beta, bf16* __restrict__ out, float* __restrict__ stats, long rows, int C,
          float eps) {
  const long row = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int nv = C / 8;
  float v[kLNMaxIter][8];
  const bf16* xr = x + row * C;
#pragma unroll
  for (int it = 0; it < kLNMaxIter; ++it) {
    const int vi = lane + it * 32;
    if (vi < nv) {
      const uint4 u = *reinterpret_cast<const uint4*>(xr + vi * 8);
      const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
      v[it][0] = a.x; v[it][1] = a.y; v[it][2] = b.x; v[it][3] = b.y;
      v[it][4] = c.x; v[it][5] = c.y; v[it][6] = d.x; v[it][7] = d.y;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[it][j] = 0.f;
    }
  }
  float mean, rstd;
  if (MODE == 0) {
    float s = 0.f;
#pragma unroll
    for (int it = 0; it < kLNMaxIter; ++it)
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[it][j];
    mean = warp_sum(s) / (float)C;
    float q = 0.f;
#pragma unroll
    for (int it = 0; it < kLNMaxIter; ++it) {
      const int vi = lane + it * 32;
      if (vi < nv) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float d = v[it][j] - mean;
          q += d * d;
        }
      }
    }
    rstd = rsqrtf(warp_sum(q) / (float)C + eps);
    if (lane == 0) {
      stats[row * 2] = mean;
      stats[row * 2 + 1] = rstd;
    }
  } else {
    mean = stats[row * 2];
    rstd = stats[row * 2 + 1];
  }
  if (MODE == 0) {
#pragma unroll
    for (int it = 0; it < kLNMaxIter; ++it) {
      const int vi = lane + it * 32;
      if (vi < nv) {
        const float4 g0 = *reinterpret_cast<const float4*>(gamma + vi * 8);
        const float4 g1 = *reinterpret_cast<const float4*>(gamma + vi * 8 + 4);
        const float4 b0 = *reinterpret_cast<const float4*>(beta + vi * 8);
        const float4 b1 = *reinterpret_cast<const float4*>(beta + vi * 8 + 4);
        const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = (v[it][j] - mean) * rstd * gg[j] + bb[j];
        *reinterpret_cast<uint4*>(out + row * C + vi * 8) =
            make_uint4(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]), pack_bf16(o[4], o[5]), pack_bf16(o[6], o[7]));
      }
    }
  } else {
    float dg[kLNMaxIter][8];
    float m1 = 0.f, m2 = 0.f;
    const bf16* dr = dy + row * C;
#pragma unroll
    for (int it = 0; it < kLNMaxIter; ++it) {
      const int vi = lane + it * 32;
      if (vi < nv) {
        const uint4 u = *reinterpret_cast<const uint4*>(dr + vi * 8);
        const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
        const float dd[8] = {a.x, a.y, b.x, b.y, c.x, c.y, d.x, d.y};
        const float4 g0 = *reinterpret_cast<const float4*>(gamma + vi * 8);
        const float4 g1 = *reinterpret_cast<const float4*>(gamma + vi * 8 + 4);
        const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = (v[it][j] - mean) * rstd;
          v[it][j] = xh;
          dg[it][j] = dd[j] * gg[j];
          m1 += dg[it][j];
          m2 += dg[it][j] * xh;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) dg[it][j] = 0.f;
      }
    }
    m1 = warp_sum(m1) / (float)C;
    m2 = warp_sum(m2) / (float)C;
#pragma unroll
    for (int it = 0; it < kLNMaxIter; ++it) {
      const int vi = lane + it * 32;
      if (vi < nv) {
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = rstd * (dg[it][j] - m1 - v[it][j] * m2);
        *reinterpret_cast<uint4*>(out + row * C + vi * 8) =
            make_uint4(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]), pack_bf16(o[4], o[5]), pack_bf16(o[6], o[7]));
      }
    }
  }
}

extern "C" int e4t_layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* stats,
                                 long long rows, int C, float eps, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  E4T_CHECK(C % 8 == 0 && C <= 2048, "e4t_layernorm_fwd: unsupported C=%d", C);
  const int it = cdiv(C, 256);
#define LN_FWD(N) ln_kernel<0, N><<<cdiv(rows, 8), 256, 0, st>>>((const bf16*)x, nullptr, gamma, beta, (bf16*)y, stats, rows, C, eps)
  if (it <= 2) LN_FWD(2); else if (it <= 3) LN_FWD(3); else if (it <= 5) LN_FWD(5); else LN_FWD(8);
#undef LN_FWD
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

extern "C" int e4t_layernorm_bwd(const void* x, const void* dy, const float* gamma, const float* stats, void* dx,
                                 long long rows, int C, float eps, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  E4T_CHECK(C % 8 == 0 && C <= 2048, "e4t_layernorm_bwd: unsupported C=%d", C);
  const int it = cdiv(C, 256);
#define LN_BWD(N) ln_kernel<1, N><<<cdiv(rows, 8), 256, 0, st>>>((const bf16*)x, (const bf16*)dy, gamma, nullptr, (bf16*)dx, const_cast<float*>(stats), rows, C, eps)
  if (it <= 2) LN_BWD(2); else if (it <= 3) LN_BWD(3); else if (it <= 5) LN_BWD(5); else LN_BWD(8);
#undef LN_BWD
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}
