// e4t_b200 — HBM-bound elementwise / small kernels of the E4T pre-training step (sm_100a).
//   WeightOffsets closed form   e4t/weightoffsets.py:14-23  (Δ = b aᵀ + s b_cᵀ + b_r 1ᵀ, SURVEY.md App. A)
//   W ⊙ (1+Δ)                   e4t/models/cross_attention.py:506,516,518
//   GEGLU                       e4t/models/attention.py:409-430
//   Upsample2D nearest x2 / stride-2 pick for Downsample2D (diffusers 0.14.0 resnet.py)
//   UNet conv_in / conv_out      e4t/models/unet_2d_condition.py:481,557
//   E4TEncoder feature mean-pool e4t/encoder.py:147-148
//   AdamW                        torch.optim.AdamW as used at pretrain_e4t.py:389-392
#include "common.cuh"

static inline int grid_for(long n, int threads) {
  long g = (n + threads - 1) / threads;
  const long cap = 148L * 32;
  return (int)(g < cap ? (g < 1 ? 1 : g) : cap);
}

// ---------------------------------------------------------------------------------------------
// GEGLU:  h [rows][2F] -> out [rows][F] = h[:, :F] * gelu(h[:, F:])   (exact erf GELU)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_f(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_grad(float x) {
  const float cdf = 0.5f * (1.f + erff(x * 0.70710678118654752f));
  const float pdf = 0.3989422804014327f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

__global__ void geglu_fwd_kernel(const bf16* __restrict__ h, bf16* __restrict__ out, long rows, int F) {
  const int vpr = F / 8;
  const long n = rows * vpr;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const long r = i / vpr;
    const int c = (int)(i % vpr) * 8;
    const uint4 u = *reinterpret_cast<const uint4*>(h + r * 2 * F + c);
    const uint4 g = *reinterpret_cast<const uint4*>(h + r * 2 * F + F + c);
    const uint32_t us[4] = {u.x, u.y, u.z, u.w}, gs[4] = {g.x, g.y, g.z, g.w};
    uint32_t os[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 a = unpack_bf16(us[j]), b = unpack_bf16(gs[j]);
      os[j] = pack_bf16(a.x * gelu_f(b.x), a.y * gelu_f(b.y));
    }
    *reinterpret_cast<uint4*>(out + r * F + c) = make_uint4(os[0], os[1], os[2], os[3]);
  }
}
__global__ void geglu_bwd_kernel(const bf16* __restrict__ h, const bf16* __restrict__ dout, bf16* __restrict__ dh,
                                 long rows, int F) {
  const int vpr = F / 8;
  const long n = rows * vpr;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const long r = i / vpr;
    const int c = (int)(i % vpr) * 8;
    const uint4 u = *reinterpret_cast<const uint4*>(h + r * 2 * F + c);
    const uint4 g = *reinterpret_cast<const uint4*>(h + r * 2 * F + F + c);
    const uint4 d = *reinterpret_cast<const uint4*>(dout + r * F + c);
    const uint32_t us[4] = {u.x, u.y, u.z, u.w}, gs[4] = {g.x, g.y, g.z, g.w}, ds[4] = {d.x, d.y, d.z, d.w};
    uint32_t ou[4], og[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 a = unpack_bf16(us[j]), b = unpack_bf16(gs[j]), dd = unpack_bf16(ds[j]);
      ou[j] = pack_bf16(dd.x * gelu_f(b.x), dd.y * gelu_f(b.y));
      og[j] = pack_bf16(dd.x * a.x * gelu_grad(b.x), dd.y * a.y * gelu_grad(b.y));
    }
    *reinterpret_cast<uint4*>(dh + r * 2 * F + c) = make_uint4(ou[0], ou[1], ou[2], ou[3]);
    *reinterpret_cast<uint4*>(dh + r * 2 * F + F + c) = make_uint4(og[0], og[1], og[2], og[3]);
  }
}
extern "C" int e4t_geglu_fwd(const void* h, void* out, long long rows, int F, void* stream_) {
  E4T_CHECK(F % 8 == 0, "e4t_geglu_fwd: F must be a multiple of 8");
  geglu_fwd_kernel<<<grid_for(rows * (F / 8), 256), 256, 0, (cudaStream_t)stream_>>>((const bf16*)h, (bf16*)out,
                                                                                     rows, F);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}
extern "C" int e4t_geglu_bwd(const void* h, const void* dout, void* dh, long long rows, int F, void* stream_) {
  E4T_CHECK(F % 8 == 0, "e4t_geglu_bwd: F must be a multiple of 8");
  geglu_bwd_kernel<<<grid_for(rows * (F / 8), 256), 256, 0, (cudaStream_t)stream_>>>(
      (const bf16*)h, (const bf16*)dout, (bf16*)dh, rows, F);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Spatial resampling on NHWC bf16 (C % 8 == 0)
//   mode 0: nearest x2 upsample   (B,H,W,C) -> (B,2H,2W,C)
//   mode 1: its adjoint           (B,2H,2W,C) -> (B,H,W,C)   (sum of the 2x2 block)
//   mode 2: stride-2 pick         (B,2H,2W,C) -> (B,H,W,C)   y[i,j] = x[2i,2j]
//   mode 3: its adjoint (zero insertion) (B,H,W,C) -> (B,2H,2W,C)
// H, W below are always the SMALL resolution.
// ---------------------------------------------------------------------------------------------
__global__ void resample_kernel(const bf16* __restrict__ x, bf16* __restrict__ y, int B, int H, int W, int C,
                                int mode) {
  const int vpc = C / 8;
  const bool out_big = (mode == 0 || mode == 3);
  const int OH = out_big ? 2 * H : H, OW = out_big ? 2 * W : W;
  const long n = (long)B * OH * OW * vpc;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const int cv = (int)(i % vpc);
    long p = i / vpc;
    const int ow = (int)(p % OW);
    p /= OW;
    const int oh = (int)(p % OH);
    const int b = (int)(p / OH);
    uint4 o;
    if (mode == 0) {
      o = *reinterpret_cast<const uint4*>(x + (((long)b * H + oh / 2) * W + ow / 2) * C + cv * 8);
    } else if (mode == 2) {
      o = *reinterpret_cast<const uint4*>(x + (((long)b * 2 * H + 2 * oh) * (2 * W) + 2 * ow) * C + cv * 8);
    } else if (mode == 3) {
      if ((oh & 1) == 0 && (ow & 1) == 0)
        o = *reinterpret_cast<const uint4*>(x + (((long)b * H + oh / 2) * W + ow / 2) * C + cv * 8);
      else
        o = make_uint4(0, 0, 0, 0);
    } else {
      float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
          const uint4 u = *reinterpret_cast<const uint4*>(
              x + (((long)b * 2 * H + 2 * oh + dy) * (2 * W) + 2 * ow + dx) * C + cv * 8);
          const float2 a = unpack_bf16(u.x), bb = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
          acc[0] += a.x; acc[1] += a.y; acc[2] += bb.x; acc[3] += bb.y;
          acc[4] += c.x; acc[5] += c.y; acc[6] += d.x; acc[7] += d.y;
        }
      o = make_uint4(pack_bf16(acc[0], acc[1]), pack_bf16(acc[2], acc[3]), pack_bf16(acc[4], acc[5]),
                     pack_bf16(acc[6], acc[7]));
    }
    *reinterpret_cast<uint4*>(y + i * 8) = o;
  }
}
extern "C" int e4t_resample2x(const void* x, void* y, int B, int H, int W, int C, int mode, void* stream_) {
  E4T_CHECK(C % 8 == 0 && mode >= 0 && mode <= 3, "e4t_resample2x: bad args");
  const bool out_big = (mode == 0 || mode == 3);
  const long n = (long)B * (out_big ? 4 : 1) * H * W * (C / 8);
  resample_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream_>>>((const bf16*)x, (bf16*)y, B, H, W, C, mode);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// WeightOffsets, closed form (R = row_dim = in_features, C = column_dim = out_features)
//   vx = w1 v + β1 (R)   vy = w2 v + β2 (C)   a = Wc vx (R)   b = Wr vy (C)   s = Wr 1 (C)
// One warp per output row; rows [0,R) produce a (and vx), rows [R,R+C) produce b, s (and vy).
// ---------------------------------------------------------------------------------------------
__global__ void wo_factors_kernel(const float* __restrict__ v, const float* __restrict__ w1,
                                  const float* __restrict__ b1, const float* __restrict__ w2,
                                  const float* __restrict__ b2, const float* __restrict__ Wc,
                                  const float* __restrict__ Wr, float* __restrict__ vx, float* __restrict__ vy,
                                  float* __restrict__ a, float* __restrict__ b, float* __restrict__ s, int R, int C) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= R + C) return;
  const float vv = v[0];
  if (row < R) {
    const float* wr = Wc + (long)row * R;
    float acc = 0.f;
    for (int j = lane; j < R; j += 32) acc += wr[j] * (w1[j] * vv + b1[j]);
    acc = warp_sum(acc);
    if (lane == 0) {
      a[row] = acc;
      vx[row] = w1[row] * vv + b1[row];
    }
  } else {
    const int c = row - R;
    const float* wr = Wr + (long)c * C;
    float acc = 0.f, sum = 0.f;
    for (int j = lane; j < C; j += 32) {
      const float w = wr[j];
      acc += w * (w2[j] * vv + b2[j]);
      sum += w;
    }
    acc = warp_sum(acc);
    sum = warp_sum(sum);
    if (lane == 0) {
      b[c] = acc;
      s[c] = sum;
      vy[c] = w2[c] * vv + b2[c];
    }
  }
}
extern "C" int e4t_wo_factors_fwd(const float* v, const float* w1, const float* b1, const float* w2, const float* b2,
                                  const float* Wc, const float* Wr, float* vx, float* vy, float* a, float* b,
                                  float* s, int R, int C, void* stream_) {
  wo_factors_kernel<<<cdiv(R + C, 8), 256, 0, (cudaStream_t)stream_>>>(v, w1, b1, w2, b2, Wc, Wr, vx, vy, a, b, s, R,
                                                                       C);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// W_eff[c][r] = bf16( W[c][r] * (1 + b[c] a[r] + s[c] bc[r] + br[c]) ),  W fp32 [C][R]
__global__ void wo_weff_kernel(const float* __restrict__ W, const float* __restrict__ a, const float* __restrict__ bc,
                               const float* __restrict__ b, const float* __restrict__ s, const float* __restrict__ br,
                               bf16* __restrict__ out, int C, int R) {
  const int vpr = R / 4;
  const long n = (long)C * vpr;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i / vpr);
    const int r = (int)(i % vpr) * 4;
    const float4 w = *reinterpret_cast<const float4*>(W + (long)c * R + r);
    const float4 av = *reinterpret_cast<const float4*>(a + r);
    const float4 bv = *reinterpret_cast<const float4*>(bc + r);
    const float bb = b[c], ss = s[c], one = 1.f + br[c];
    const float o0 = w.x * (one + bb * av.x + ss * bv.x), o1 = w.y * (one + bb * av.y + ss * bv.y);
    const float o2 = w.z * (one + bb * av.z + ss * bv.z), o3 = w.w * (one + bb * av.w + ss * bv.w);
    *reinterpret_cast<uint2*>(out + (long)c * R + r) = make_uint2(pack_bf16(o0, o1), pack_bf16(o2, o3));
  }
}
extern "C" int e4t_wo_weff_fwd(const float* W, const float* a, const float* bc, const float* b, const float* s,
                               const float* br, void* w_eff, int C, int R, void* stream_) {
  E4T_CHECK(R % 4 == 0, "e4t_wo_weff_fwd: R must be a multiple of 4");
  wo_weff_kernel<<<grid_for((long)C * R / 4, 256), 256, 0, (cudaStream_t)stream_>>>(W, a, bc, b, s, br, (bf16*)w_eff,
                                                                                    C, R);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// Backward reductions of G = dW_eff ⊙ W  (dW_eff fp32 [C][R], accumulated by the split-K weight-grad GEMM):
//   Ga[c] = Σ_r G a[r]   Gbc[c] = Σ_r G bc[r]   G1[c] = Σ_r G        (row reductions)
//   GTb[r] = Σ_c G b[c]  GTs[r] = Σ_c G s[c]                          (column reductions, atomics; pre-zeroed)
// One CTA = 8 rows (one warp per row).
__global__ void __launch_bounds__(256)
wo_bwd_reduce_kernel(const float* __restrict__ dWeff, const float* __restrict__ W, const float* __restrict__ a,
                     const float* __restrict__ bc, const float* __restrict__ b, const float* __restrict__ s,
                     float* __restrict__ Ga, float* __restrict__ Gbc, float* __restrict__ G1,
                     float* __restrict__ GTb, float* __restrict__ GTs, int C, int R) {
  extern __shared__ float wsm[];  // [2][R] column partials
  float* cb = wsm;
  float* cs = wsm + R;
  for (int r = threadIdx.x; r < R; r += blockDim.x) cb[r] = cs[r] = 0.f;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * 8 + warp;
  if (c < C) {
    const float bcv = b[c], scv = s[c];
    float ga = 0.f, gbc = 0.f, g1 = 0.f;
    for (int r = lane; r < R; r += 32) {
      const float g = dWeff[(long)c * R + r] * W[(long)c * R + r];
      ga += g * a[r];
      gbc += g * bc[r];
      g1 += g;
      atomicAdd(&cb[r], g * bcv);
      atomicAdd(&cs[r], g * scv);
    }
    ga = warp_sum(ga);
    gbc = warp_sum(gbc);
    g1 = warp_sum(g1);
    if (lane == 0) {
      Ga[c] = ga;
      Gbc[c] = gbc;
      G1[c] = g1;
    }
  }
  __syncthreads();
  for (int r = threadIdx.x; r < R; r += blockDim.x) {
    atomicAdd(&GTb[r], cb[r]);
    atomicAdd(&GTs[r], cs[r]);
  }
}
// Column mat-vec: out[j] += Σ_{i in chunk} M[i][j] x[i]   (M [n][n] row-major; out pre-zeroed)
// grid (n/128 column tiles, row chunks of 32); coalesced over j, one atomic per (thread, chunk).
__global__ void colmatvec_kernel(const float* __restrict__ M, const float* __restrict__ x, float* __restrict__ out,
                                 int n) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i0 = blockIdx.y * 32;
  if (j >= n) return;
  float acc = 0.f;
  const int i1 = min(n, i0 + 32);
#pragma unroll 8
  for (int i = i0; i < i1; ++i) acc += M[(long)i * n + j] * x[i];
  atomicAdd(&out[j], acc);
}
// dM[i][j] = u[i] * w[j] + (t ? t[i] : 0)
__global__ void outer_kernel(const float* __restrict__ u, const float* __restrict__ w, const float* __restrict__ t,
                             float* __restrict__ dM, int n) {
  const long total = (long)n * n;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int r = (int)(i / n), c = (int)(i % n);
    dM[i] = u[r] * w[c] + (t ? t[r] : 0.f);
  }
}
// dw = dvec*v ; dbeta = dvec ; dv_part = Σ w*dvec  (one block)
__global__ void wo_vec_grads_kernel(const float* __restrict__ dvx, const float* __restrict__ dvy,
                                    const float* __restrict__ w1, const float* __restrict__ w2,
                                    const float* __restrict__ v, float* __restrict__ dw1, float* __restrict__ db1,
                                    float* __restrict__ dw2, float* __restrict__ db2, float* __restrict__ dv, int R,
                                    int C) {
  __shared__ float red[32];
  const float vv = v[0];
  float acc = 0.f;
  for (int j = threadIdx.x; j < R; j += blockDim.x) {
    const float d = dvx[j];
    dw1[j] = d * vv;
    db1[j] = d;
    acc += w1[j] * d;
  }
  for (int j = threadIdx.x; j < C; j += blockDim.x) {
    const float d = dvy[j];
    dw2[j] = d * vv;
    db2[j] = d;
    acc += w2[j] * d;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) dv[0] = t;
  }
}
// Full WeightOffsets backward from the accumulated dW_eff.  scratch: fp32 [3C + 2R + R + C] = Ga,Gbc,G1,GTb,GTs,dvx,dvy
// Gradient outputs are WRITTEN (not accumulated): dv[1], dw1[R], db1[R], dw2[C], db2[C], dWc[R][R], dbc[R], dWr[C][C], dbr[C]
extern "C" int e4t_wo_bwd(const float* dWeff, const float* W, const float* v, const float* w1, const float* w2,
                          const float* Wc, const float* Wr, const float* bc, const float* vx, const float* vy,
                          const float* a, const float* b, const float* s, float* scratch, float* dv, float* dw1,
                          float* db1, float* dw2, float* db2, float* dWc, float* dbc, float* dWr, float* dbr, int R,
                          int C, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  float* Ga = scratch;
  float* Gbc = Ga + C;
  float* G1 = Gbc + C;
  float* GTb = G1 + C;
  float* GTs = GTb + R;
  float* dvx = GTs + R;
  float* dvy = dvx + R;
  E4T_CUDA(cudaMemsetAsync(GTb, 0, (size_t)(2 * R + R + C) * sizeof(float), st));  // GTb, GTs, dvx, dvy
  wo_bwd_reduce_kernel<<<cdiv(C, 8), 256, (size_t)2 * R * sizeof(float), st>>>(dWeff, W, a, bc, b, s, Ga, Gbc, G1, GTb,
                                                                               GTs, C, R);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  // dWr = Ga vyᵀ + Gbc 1ᵀ ; dbr = G1
  outer_kernel<<<grid_for((long)C * C, 256), 256, 0, st>>>(Ga, vy, Gbc, dWr, C);
  E4T_COUNT_LAUNCH();
  E4T_CUDA(cudaMemcpyAsync(dbr, G1, (size_t)C * sizeof(float), cudaMemcpyDeviceToDevice, st));
  // dWc = GTb vxᵀ ; dbc = GTs
  outer_kernel<<<grid_for((long)R * R, 256), 256, 0, st>>>(GTb, vx, nullptr, dWc, R);
  E4T_COUNT_LAUNCH();
  E4T_CUDA(cudaMemcpyAsync(dbc, GTs, (size_t)R * sizeof(float), cudaMemcpyDeviceToDevice, st));
  // dvy = Wrᵀ Ga ; dvx = Wcᵀ GTb
  colmatvec_kernel<<<dim3(cdiv(C, 128), cdiv(C, 32)), 128, 0, st>>>(Wr, Ga, dvy, C);
  E4T_COUNT_LAUNCH();
  colmatvec_kernel<<<dim3(cdiv(R, 128), cdiv(R, 32)), 128, 0, st>>>(Wc, GTb, dvx, R);
  E4T_COUNT_LAUNCH();
  wo_vec_grads_kernel<<<1, 256, 0, st>>>(dvx, dvy, w1, w2, v, dw1, db1, dw2, db2, dv, R, C);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Mean-pool of a feature map (B,HW,C) bf16 -> out[b][c_off + c] fp32 (row stride ldo), and its adjoint.
// ---------------------------------------------------------------------------------------------
__global__ void meanpool_fwd_kernel(const bf16* __restrict__ x, float* __restrict__ out, int HW, int C, int ldo,
                                    int c_off) {
  // grid (C/64 chunks, B); block 256 = 32 channel-pairs x 8 row lanes
  __shared__ float2 red[8][32];
  const int b = blockIdx.y;
  const int cp = blockIdx.x * 32 + (threadIdx.x & 31);  // channel pair
  const int rl = threadIdx.x >> 5;
  float s0 = 0.f, s1 = 0.f;
  if (cp * 2 < C) {
    const uint32_t* xp = reinterpret_cast<const uint32_t*>(x + (long)b * HW * C) + cp;
    for (int r = rl; r < HW; r += 8) {
      const float2 v = unpack_bf16(xp[(long)r * (C / 2)]);
      s0 += v.x;
      s1 += v.y;
    }
  }
  red[rl][threadIdx.x & 31] = make_float2(s0, s1);
  __syncthreads();
  if (rl == 0 && cp * 2 < C) {
    float t0 = 0.f, t1 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      t0 += red[i][threadIdx.x].x;
      t1 += red[i][threadIdx.x].y;
    }
    out[(long)b * ldo + c_off + cp * 2] = t0 / (float)HW;
    out[(long)b * ldo + c_off + cp * 2 + 1] = t1 / (float)HW;
  }
}
__global__ void meanpool_bwd_kernel(const float* __restrict__ dout, bf16* __restrict__ dx, int B, int HW, int C,
                                    int ldo, int c_off) {
  const int vpr = C / 8;
  const long n = (long)B * HW * vpr;
  const float inv = 1.f / (float)HW;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % vpr) * 8;
    const int b = (int)(i / ((long)HW * vpr));
    const float* d = dout + (long)b * ldo + c_off + c;
    *reinterpret_cast<uint4*>(dx + i * 8) =
        make_uint4(pack_bf16(d[0] * inv, d[1] * inv), pack_bf16(d[2] * inv, d[3] * inv),
                   pack_bf16(d[4] * inv, d[5] * inv), pack_bf16(d[6] * inv, d[7] * inv));
  }
}
extern "C" int e4t_meanpool_fwd(const void* x, float* out, int B, int HW, int C, int ldo, int c_off, void* stream_) {
  E4T_CHECK(C % 2 == 0, "e4t_meanpool_fwd: C must be even");
  meanpool_fwd_kernel<<<dim3(cdiv(C, 64), B), 256, 0, (cudaStream_t)stream_>>>((const bf16*)x, out, HW, C, ldo, c_off);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}
extern "C" int e4t_meanpool_bwd(const float* dout, void* dx, int B, int HW, int C, int ldo, int c_off,
                                void* stream_) {
  E4T_CHECK(C % 8 == 0, "e4t_meanpool_bwd: C must be a multiple of 8");
  meanpool_bwd_kernel<<<grid_for((long)B * HW * C / 8, 256), 256, 0, (cudaStream_t)stream_>>>(dout, (bf16*)dx, B, HW,
                                                                                              C, ldo, c_off);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// conv_in: NCHW fp32 (B,Cin<=8,H,W) -> NHWC bf16 (B,H,W,Cout), 3x3 pad 1.  w fp32 [Cout][Cin][3][3].
// ---------------------------------------------------------------------------------------------
__global__ void conv_in_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                               bf16* __restrict__ y, int B, int Cin, int H, int W, int Cout) {
  // one CTA per (b, h, 8-pixel strip); threads over Cout
  extern __shared__ float cin_sm[];  // [Cin][3][10] input patch
  const int strips = W / 8;
  const int w0 = (blockIdx.x % strips) * 8;
  const int h = (blockIdx.x / strips) % H;
  const int b = blockIdx.x / (strips * H);
  for (int i = threadIdx.x; i < Cin * 30; i += blockDim.x) {
    const int ci = i / 30, rr = (i % 30) / 10, cc = i % 10;
    const int hh = h + rr - 1, ww = w0 + cc - 1;
    cin_sm[i] = (hh >= 0 && hh < H && ww >= 0 && ww < W) ? x[(((long)b * Cin + ci) * H + hh) * W + ww] : 0.f;
  }
  __syncthreads();
  for (int co = threadIdx.x; co < Cout; co += blockDim.x) {
    float acc[8];
    const float bv = bias ? bias[co] : 0.f;
#pragma unroll
    for (int p = 0; p < 8; ++p) acc[p] = bv;
    for (int ci = 0; ci < Cin; ++ci)
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float wv = w[((long)co * Cin + ci) * 9 + ky * 3 + kx];
#pragma unroll
          for (int p = 0; p < 8; ++p) acc[p] += wv * cin_sm[ci * 30 + ky * 10 + p + kx];
        }
#pragma unroll
    for (int p = 0; p < 8; ++p) y[(((long)b * H + h) * W + w0 + p) * Cout + co] = __float2bfloat16(acc[p]);
  }
}
extern "C" int e4t_conv_in_fwd(const float* x, const float* w, const float* bias, void* y, int B, int Cin, int H,
                               int W, int Cout, void* stream_) {
  E4T_CHECK(W % 8 == 0 && Cin <= 16, "e4t_conv_in_fwd: W %% 8 != 0 or Cin > 16");
  conv_in_kernel<<<B * H * (W / 8), 128, (size_t)Cin * 30 * sizeof(float), (cudaStream_t)stream_>>>(x, w, bias, (bf16*)y,
                                                                                                   B, Cin, H, W, Cout);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// 1x1 convolution on NCHW fp32, y[b][o][p] = bias[o] + sum_i w[o][i] x[b][i][p] (Cin, Cout <= 8): the VAE's
// post_quant_conv on the latents, applied on its own so that the decoder's conv_in zero-pads the transformed latents.
__global__ void pointwise_nchw_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                      const float* __restrict__ bias, float* __restrict__ y, int B, int Cin, int Cout,
                                      long HW) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < (long)B * HW; i += (long)gridDim.x * blockDim.x) {
    const long b = i / HW, p = i % HW;
    float xv[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) xv[c] = c < Cin ? x[(b * Cin + c) * HW + p] : 0.f;
    for (int o = 0; o < Cout; ++o) {
      float acc = bias ? bias[o] : 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c)
        if (c < Cin) acc = fmaf(w[o * Cin + c], xv[c], acc);
      y[(b * Cout + o) * HW + p] = acc;
    }
  }
}
extern "C" int e4t_pointwise_nchw(const float* x, const float* w, const float* bias, float* y, int B, int Cin, int Cout,
                                  long long HW, void* stream_) {
  E4T_CHECK(Cin >= 1 && Cin <= 8 && Cout >= 1 && Cout <= 8, "e4t_pointwise_nchw: Cin, Cout must be in [1, 8]");
  pointwise_nchw_kernel<<<grid_for((long)B * HW, 256), 256, 0, (cudaStream_t)stream_>>>(x, w, bias, y, B, Cin, Cout,
                                                                                       (long)HW);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// conv_out: NHWC bf16 (B,H,W,C) -> NCHW fp32 (B,Cout<=8,H,W); w fp32 [Cout][C][3][3].  One warp per pixel.
__global__ void conv_out_fwd_kernel(const bf16* __restrict__ x, const float* __restrict__ w,
                                    const float* __restrict__ bias, float* __restrict__ y, int B, int H, int W, int C,
                                    int Cout) {
  const long pix = (long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pix >= (long)B * H * W) return;
  const int ww = (int)(pix % W), hh = (int)((pix / W) % H), b = (int)(pix / ((long)W * H));
  float acc[8];
#pragma unroll
  for (int o = 0; o < 8; ++o) acc[o] = 0.f;
  for (int ky = 0; ky < 3; ++ky) {
    const int ih = hh + ky - 1;
    if (ih < 0 || ih >= H) continue;
    for (int kx = 0; kx < 3; ++kx) {
      const int iw = ww + kx - 1;
      if (iw < 0 || iw >= W) continue;
      const bf16* xp = x + (((long)b * H + ih) * W + iw) * C;
      for (int c = lane; c < C; c += 32) {
        const float xv = __bfloat162float(xp[c]);
#pragma unroll
        for (int o = 0; o < 8; ++o)
          if (o < Cout) acc[o] += xv * w[((long)o * C + c) * 9 + ky * 3 + kx];
      }
    }
  }
#pragma unroll
  for (int o = 0; o < 8; ++o) {
    if (o < Cout) {
      const float t = warp_sum(acc[o]);
      if (lane == 0) y[(((long)b * Cout + o) * H + hh) * W + ww] = t + (bias ? bias[o] : 0.f);
    }
  }
}
// dx[b,h,w,c] = Σ_o Σ_taps w[o][c][ky][kx] * dy[b,o,h-ky+1,w-kx+1]   -> NHWC bf16
__global__ void conv_out_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ w, bf16* __restrict__ dx,
                                    int B, int H, int W, int C, int Cout) {
  const long n = (long)B * H * W * C;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    long p = i / C;
    const int ww = (int)(p % W);
    p /= W;
    const int hh = (int)(p % H);
    const int b = (int)(p / H);
    float acc = 0.f;
    for (int o = 0; o < Cout; ++o)
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const int oh = hh - ky + 1;
        if (oh < 0 || oh >= H) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int ow = ww - kx + 1;
          if (ow < 0 || ow >= W) continue;
          acc += w[((long)o * C + c) * 9 + ky * 3 + kx] * dy[(((long)b * Cout + o) * H + oh) * W + ow];
        }
      }
    dx[i] = __float2bfloat16(acc);
  }
}
extern "C" int e4t_conv_out_fwd(const void* x, const float* w, const float* bias, float* y, int B, int H, int W, int C,
                                int Cout, void* stream_) {
  E4T_CHECK(Cout <= 8, "e4t_conv_out_fwd: Cout must be <= 8");
  conv_out_fwd_kernel<<<cdiv((long)B * H * W, 8), 256, 0, (cudaStream_t)stream_>>>((const bf16*)x, w, bias, y, B, H, W,
                                                                                   C, Cout);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}
extern "C" int e4t_conv_out_bwd(const float* dy, const float* w, void* dx, int B, int H, int W, int C, int Cout,
                                void* stream_) {
  conv_out_bwd_kernel<<<grid_for((long)B * H * W * C, 256), 256, 0, (cudaStream_t)stream_>>>(dy, w, (bf16*)dx, B, H, W,
                                                                                             C, Cout);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Fused AdamW over a flat fp32 parameter arena (torch.optim.AdamW semantics, amsgrad=False).
// ---------------------------------------------------------------------------------------------
__global__ void adamw_tick_kernel(int* step) { *step += 1; }
__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                             float* __restrict__ v, long n, float lr, float beta1, float beta2, float eps, float wd,
                             const int* __restrict__ step_ptr, int step_host, float grad_scale) {
  // bias corrections from the DEVICE step counter when given (CUDA-graph replays advance it), else the host value
  const int step = step_ptr ? *step_ptr : step_host;
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2_sqrt = sqrtf(1.f - powf(beta2, (float)step));
  const long n4 = n / 4;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    float4 pp = reinterpret_cast<float4*>(p)[i];
    const float4 gg = reinterpret_cast<const float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
    float* pa = &pp.x;
    const float* ga = &gg.x;
    float* ma = &mm.x;
    float* va = &vv.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float gr = ga[j] * grad_scale;
      pa[j] *= (1.f - lr * wd);
      ma[j] = beta1 * ma[j] + (1.f - beta1) * gr;
      va[j] = beta2 * va[j] + (1.f - beta2) * gr * gr;
      const float denom = sqrtf(va[j]) / bc2_sqrt + eps;
      pa[j] -= (lr / bc1) * ma[j] / denom;
    }
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
  }
  for (long i = n4 * 4 + (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float gr = g[i] * grad_scale;
    float pv = p[i] * (1.f - lr * wd);
    const float mv = beta1 * m[i] + (1.f - beta1) * gr;
    const float vv2 = beta2 * v[i] + (1.f - beta2) * gr * gr;
    pv -= (lr / bc1) * mv / (sqrtf(vv2) / bc2_sqrt + eps);
    p[i] = pv;
    m[i] = mv;
    v[i] = vv2;
  }
}
extern "C" int e4t_adamw_step(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                              float beta2, float eps, float weight_decay, int step, float grad_scale, void* stream_) {
  E4T_CHECK(((uintptr_t)p % 16) == 0 && ((uintptr_t)g % 16) == 0 && ((uintptr_t)m % 16) == 0 && ((uintptr_t)v % 16) == 0,
            "e4t_adamw_step: buffers must be 16-byte aligned");
  adamw_kernel<<<grid_for(n / 4 + 1, 256), 256, 0, (cudaStream_t)stream_>>>(p, g, m, v, n, lr, beta1, beta2, eps,
                                                                            weight_decay, nullptr, step, grad_scale);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}
// Same, with the step counter in device memory: *step_dev is incremented, then used (CUDA-graph friendly).
extern "C" int e4t_adamw_step_dev(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                                  float beta2, float eps, float weight_decay, int* step_dev, float grad_scale,
                                  void* stream_) {
  E4T_CHECK(((uintptr_t)p % 16) == 0 && ((uintptr_t)g % 16) == 0 && ((uintptr_t)m % 16) == 0 && ((uintptr_t)v % 16) == 0,
            "e4t_adamw_step_dev: buffers must be 16-byte aligned");
  adamw_tick_kernel<<<1, 1, 0, (cudaStream_t)stream_>>>(step_dev);
  E4T_COUNT_LAUNCH();
  adamw_kernel<<<grid_for(n / 4 + 1, 256), 256, 0, (cudaStream_t)stream_>>>(p, g, m, v, n, lr, beta1, beta2, eps,
                                                                            weight_decay, step_dev, 0, grad_scale);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------
// WeightOffsets BANK: the same kernels as above, batched over ALL projections of a UNet (96 for SD-v1.4) so that
// a step needs 2 forward + 5 backward launches instead of ~1000 tiny ones.  `tab` is a device array of WOProj
// (one per projection), built once by the host binding from the module tree.
// ---------------------------------------------------------------------------------------------
struct WOProj {
  const float *W, *v, *w1, *b1, *w2, *b2, *Wc, *bc, *Wr, *br;  // parameters (fp32)
  float* fac;      // forward scratch : vx[R] a[R] vy[C] b[C] s[C]
  float* bw;       // backward scratch: Ga[C] Gbc[C] G1[C] GTb[R] GTs[R] dvx[R] dvy[C]   (zeroed per backward)
  bf16* weff;      // [C][R] slice of the fused W_eff storage
  const float* dweff;  // [C][R] slice of the accumulated weight gradient
  float *dv, *dw1, *db1, *dw2, *db2, *dWc, *dbc, *dWr, *dbr;  // gradient destinations (written)
  int R, C;
};
__device__ __forceinline__ float* wo_vx(const WOProj& p) { return p.fac; }
__device__ __forceinline__ float* wo_a(const WOProj& p) { return p.fac + p.R; }
__device__ __forceinline__ float* wo_vy(const WOProj& p) { return p.fac + 2 * p.R; }
__device__ __forceinline__ float* wo_b(const WOProj& p) { return p.fac + 2 * p.R + p.C; }
__device__ __forceinline__ float* wo_s(const WOProj& p) { return p.fac + 2 * p.R + 2 * p.C; }
__device__ __forceinline__ float* wo_bw(const WOProj& p) { return p.bw; }

__global__ void wo_bank_factors_kernel(const WOProj* __restrict__ tab) {
  const WOProj p = tab[blockIdx.y];
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= p.R + p.C) return;
  const float vv = p.v[0];
  if (row < p.R) {
    const float* wr = p.Wc + (long)row * p.R;
    float acc = 0.f;
    for (int j = lane; j < p.R; j += 32) acc += wr[j] * (p.w1[j] * vv + p.b1[j]);
    acc = warp_sum(acc);
    if (lane == 0) {
      wo_a(p)[row] = acc;
      wo_vx(p)[row] = p.w1[row] * vv + p.b1[row];
    }
  } else {
    const int c = row - p.R;
    const float* wr = p.Wr + (long)c * p.C;
    float acc = 0.f, sum = 0.f;
    for (int j = lane; j < p.C; j += 32) {
      const float w = wr[j];
      acc += w * (p.w2[j] * vv + p.b2[j]);
      sum += w;
    }
    acc = warp_sum(acc);
    sum = warp_sum(sum);
    if (lane == 0) {
      wo_b(p)[c] = acc;
      wo_s(p)[c] = sum;
      wo_vy(p)[c] = p.w2[c] * vv + p.b2[c];
    }
  }
}
__global__ void wo_bank_weff_kernel(const WOProj* __restrict__ tab) {
  const WOProj p = tab[blockIdx.y];
  const int vpr = p.R / 4;
  const long n = (long)p.C * vpr;
  const float* a = wo_a(p);
  const float* b = wo_b(p);
  const float* s = wo_s(p);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i / vpr);
    const int r = (int)(i % vpr) * 4;
    const float4 w = *reinterpret_cast<const float4*>(p.W + (long)c * p.R + r);
    const float4 av = *reinterpret_cast<const float4*>(a + r);
    const float4 bv = *reinterpret_cast<const float4*>(p.bc + r);
    const float bb = b[c], ss = s[c], one = 1.f + p.br[c];
    *reinterpret_cast<uint2*>(p.weff + (long)c * p.R + r) =
        make_uint2(pack_bf16(w.x * (one + bb * av.x + ss * bv.x), w.y * (one + bb * av.y + ss * bv.y)),
                   pack_bf16(w.z * (one + bb * av.z + ss * bv.z), w.w * (one + bb * av.w + ss * bv.w)));
  }
}
// backward 1: row / column reductions of G = dW_eff ⊙ W  (GTb, GTs pre-zeroed)
__global__ void __launch_bounds__(256) wo_bank_reduce_kernel(const WOProj* __restrict__ tab) {
  const WOProj p = tab[blockIdx.y];
  extern __shared__ float wsm[];  // [2][Rmax]
  if (blockIdx.x * 8 >= p.C) return;
  const int R = p.R, C = p.C;
  float* cb = wsm;
  float* cs = wsm + R;
  for (int r = threadIdx.x; r < R; r += blockDim.x) cb[r] = cs[r] = 0.f;
  __syncthreads();
  const float* a = wo_a(p);
  const float* b = wo_b(p);
  const float* s = wo_s(p);
  float* bw = wo_bw(p);
  float *Ga = bw, *Gbc = bw + C, *G1 = bw + 2 * C, *GTb = bw + 3 * C, *GTs = bw + 3 * C + R;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * 8 + warp;
  if (c < C) {
    const float bcv = b[c], scv = s[c];
    float ga = 0.f, gbc = 0.f, g1 = 0.f;
    for (int r = lane; r < R; r += 32) {
      const float g = p.dweff[(long)c * R + r] * p.W[(long)c * R + r];
      ga += g * a[r];
      gbc += g * p.bc[r];
      g1 += g;
      atomicAdd(&cb[r], g * bcv);
      atomicAdd(&cs[r], g * scv);
    }
    ga = warp_sum(ga);
    gbc = warp_sum(gbc);
    g1 = warp_sum(g1);
    if (lane == 0) {
      Ga[c] = ga;
      Gbc[c] = gbc;
      G1[c] = g1;
    }
  }
  __syncthreads();
  for (int r = threadIdx.x; r < R; r += blockDim.x) {
    atomicAdd(&GTb[r], cb[r]);
    atomicAdd(&GTs[r], cs[r]);
  }
}
// backward 2: dvy = Wrᵀ Ga, dvx = Wcᵀ GTb (column mat-vecs; dvx/dvy pre-zeroed).  blockIdx.z = 2*proj + which
__global__ void wo_bank_colmatvec_kernel(const WOProj* __restrict__ tab) {
  const WOProj p = tab[blockIdx.z >> 1];
  const int which = blockIdx.z & 1;  // 0: Wr/Ga -> dvy (n = C), 1: Wc/GTb -> dvx (n = R)
  const int n = which == 0 ? p.C : p.R;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i0 = blockIdx.y * 32;
  if (j >= n || i0 >= n) return;
  float* bw = wo_bw(p);
  const float* M = which == 0 ? p.Wr : p.Wc;
  const float* x = which == 0 ? bw : bw + 3 * p.C;
  float* out = which == 0 ? bw + 3 * p.C + 3 * p.R : bw + 3 * p.C + 2 * p.R;
  float acc = 0.f;
  const int i1 = min(n, i0 + 32);
#pragma unroll 8
  for (int i = i0; i < i1; ++i) acc += M[(long)i * n + j] * x[i];
  atomicAdd(&out[j], acc);
}
// backward 3: dWr = Ga vyᵀ + Gbc 1ᵀ, dWc = GTb vxᵀ.  blockIdx.y = 2*proj + which
__global__ void wo_bank_outer_kernel(const WOProj* __restrict__ tab) {
  const WOProj p = tab[blockIdx.y >> 1];
  const int which = blockIdx.y & 1;
  float* bw = wo_bw(p);
  const int n = which == 0 ? p.C : p.R;
  const float* u = which == 0 ? bw : bw + 3 * p.C;                 // Ga | GTb
  const float* w = which == 0 ? wo_vy(p) : wo_vx(p);
  const float* t = which == 0 ? bw + p.C : nullptr;               // Gbc
  float* dM = which == 0 ? p.dWr : p.dWc;
  const long total = (long)n * n / 4;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int r = (int)((i * 4) / n), c = (int)((i * 4) % n);
    const float ur = u[r], tr = t ? t[r] : 0.f;
    const float4 wv = *reinterpret_cast<const float4*>(w + c);
    // ACCUMULATE into the .grad view (zeroed by zero_grad): several backward passes before an optimiser step
    // (gradient accumulation, accelerator.accumulate in pretrain_e4t.py:595) add up like torch's AccumulateGrad
    float4 g = *reinterpret_cast<const float4*>(dM + i * 4);
    g.x += ur * wv.x + tr; g.y += ur * wv.y + tr; g.z += ur * wv.z + tr; g.w += ur * wv.w + tr;
    *reinterpret_cast<float4*>(dM + i * 4) = g;
  }
}
// backward 4: vector grads (dw1, db1, dw2, db2, dv) and dbr += G1, dbc += GTs (accumulating).  one block per projection
__global__ void wo_bank_vec_kernel(const WOProj* __restrict__ tab) {
  const WOProj p = tab[blockIdx.x];
  __shared__ float red[32];
  const int R = p.R, C = p.C;
  float* bw = wo_bw(p);
  const float *G1 = bw + 2 * C, *GTs = bw + 3 * C + R, *dvx = bw + 3 * C + 2 * R, *dvy = bw + 3 * C + 3 * R;
  const float vv = p.v[0];
  float acc = 0.f;
  for (int j = threadIdx.x; j < R; j += blockDim.x) {
    const float d = dvx[j];
    p.dw1[j] += d * vv;
    p.db1[j] += d;
    p.dbc[j] += GTs[j];
    acc += p.w1[j] * d;
  }
  for (int j = threadIdx.x; j < C; j += blockDim.x) {
    const float d = dvy[j];
    p.dw2[j] += d * vv;
    p.db2[j] += d;
    p.dbr[j] += G1[j];
    acc += p.w2[j] * d;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
    if (threadIdx.x == 0) p.dv[0] += t;
  }
}
// tab: device array of n WOProj records; max_r / max_c: largest row/column dims in the bank.
extern "C" int e4t_wo_bank_fwd(const void* tab, int n, int max_r, int max_c, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const WOProj* t = (const WOProj*)tab;
  wo_bank_factors_kernel<<<dim3(cdiv(max_r + max_c, 8), n), 256, 0, st>>>(t);
  E4T_COUNT_LAUNCH();
  wo_bank_weff_kernel<<<dim3(cdiv((long)max_r * max_c / 4, 256 * 4), n), 256, 0, st>>>(t);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}
// fac_bw: pointer to the start of the (contiguous) factor scratch of the whole bank and its size in floats: the
// backward sub-ranges that need zeroing (GTb, GTs, dvx, dvy) are zeroed by clearing every projection's backward area.
// Phase 1: G reductions.  bw of every projection then holds Ga[C] Gbc[C] G1[C] GTb[R] GTs[R] (and zeros for dvx, dvy).
// Everything after this point is LINEAR in these five vectors with coefficients that depend on the parameters only, so a
// data-parallel run may all-reduce the (contiguous, ~2 MB) bw buffer here instead of the 573 MB of parameter gradients.
extern "C" int e4t_wo_bank_bwd_reduce(const void* tab, int n, int max_r, int max_c, float* bw_base, long long bw_floats,
                                      void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const WOProj* t = (const WOProj*)tab;
  E4T_CUDA(cudaMemsetAsync(bw_base, 0, (size_t)bw_floats * sizeof(float), st));
  wo_bank_reduce_kernel<<<dim3(cdiv(max_c, 8), n), 256, (size_t)2 * max_r * sizeof(float), st>>>(t);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}
// Phase 2: parameter gradients from the (possibly all-reduced) five vectors, accumulated into the .grad views.
extern "C" int e4t_wo_bank_bwd_apply(const void* tab, int n, int max_r, int max_c, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const WOProj* t = (const WOProj*)tab;
  const int mx = max_r > max_c ? max_r : max_c;
  wo_bank_colmatvec_kernel<<<dim3(cdiv(mx, 128), cdiv(mx, 32), 2 * n), 128, 0, st>>>(t);
  E4T_COUNT_LAUNCH();
  wo_bank_outer_kernel<<<dim3(cdiv((long)mx * mx / 4, 256 * 4), 2 * n), 256, 0, st>>>(t);
  E4T_COUNT_LAUNCH();
  wo_bank_vec_kernel<<<n, 256, 0, st>>>(t);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}
extern "C" int e4t_wo_bank_bwd(const void* tab, int n, int max_r, int max_c, float* bw_base, long long bw_floats,
                               void* stream_) {
  if (int e = e4t_wo_bank_bwd_reduce(tab, n, max_r, max_c, bw_base, bw_floats, stream_)) return e;
  return e4t_wo_bank_bwd_apply(tab, n, max_r, max_c, stream_);
}
extern "C" int e4t_wo_bank_record_size(void) { return (int)sizeof(WOProj); }
