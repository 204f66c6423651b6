// e4t_b200 — tcgen05 GEMM engine (sm_100a).
//
// One persistent, warp-specialised kernel serves every dense contraction on the E4T hot path:
//   * linear layers   Y[M,N] = A[M,K] · B[N,K]^T            (both operands K-major, e.g. F.linear;
//                                                            reference call sites cross_attention.py:506-518,534,
//                                                            attention.py:429 (GEGLU proj), transformer_2d.py proj_in/out)
//   * weight-gradient  dW[C,R] = dY[m,C]^T · X[m,R]          (both operands MN-major, split-K, fp32 atomic accumulate)
//   * input-gradient   dX[M,K] = dY[M,N] · W[N,K]            (A K-major, B MN-major)
//   * 3x3 convolution  (implicit GEMM over NHWC, 9 taps x Cin/64 K-chunks, halo by TMA out-of-bounds zero fill;
//                       diffusers ResnetBlock2D conv1/conv2, Upsample2D.conv, Downsample2D.conv)
//
// Structure (per CTA, 256 threads): warp0 = TMA producer, warp1 = MMA issuer (one thread issues tcgen05.mma),
// warp2 = TMEM allocator, warps4-7 = epilogue (TMEM -> registers -> global).  smem ring of `stages`
// {A 128x64, B BNx64} bf16 tiles (SWIZZLE_128B), two TMEM accumulator stages of 256 columns so the epilogue of
// tile i overlaps the MMAs of tile i+1.
#include "common.cuh"
#include <stdlib.h>

struct GemmArgs {
  int M, N, K, batch;
  int BN, m_tiles, n_tiles, splits, kchunks, kper, stages;
  int a_mn, b_mn, a_batched, b_batched;
  // implicit 3x3 convolution (conv = 1: forward / dgrad, 2: weight gradient)
  int conv, H, W, BH, BB, cin_chunks, cout;
  int cstride;   // spatial stride of the forward convolution (1, or 2 = Downsample2D; H, W are the OUTPUT size)
  int cpad;      // top/left zero padding of the forward convolution (1, or 0 = the VAE's F.pad(x, (0,1,0,1)) downsample)
  // epilogue
  void* out;
  int out_mode;  // 0 = bf16 store, 1 = fp32 store, 2 = fp32 atomic add
  long long ldo, out_bstride;
  const float* bias;      // [N] or null
  const float* rowgroup;  // [M / rows_per_group][N] fp32 (e.g. time-embedding add per image) or null
  int rows_per_group;
  const bf16* residual;  // [M][ldr] bf16 or null
  long long ldr, res_bstride;
  float alpha;
  int debug;      // E4T_GEMM_DEBUG probes: 1 skip epilogue body, 4 skip output staging, 8 no TMA loads, 16 no MMAs
  int tma_store;  // bf16 output through smem staging + TMA store (coalesced, asynchronous)
  int epi_plain;  // default on (E4T_GEMM_EPI_PLAIN=0 disables): separate slab loop for outputs without alpha/bias/rowgroup/residual
  int epi_vec;    // the per-thread epilogue's 16-byte accesses (output, residual, row-group rows) are aligned; else scalar
};

static constexpr int kBM = 128;
static constexpr int kBK = 64;
static constexpr int kATileBytes = kBM * kBK * 2;  // 16 KiB
static constexpr int kThreads = 384;  // 4 role warps + 8 epilogue warps (2 column halves x 4 lane quadrants)
static constexpr int kCSlabs = 4;  // output staging slabs (8 KiB each) for the TMA-store epilogue

__global__ void __launch_bounds__(kThreads, 1)
e4t_gemm_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                const __grid_constant__ CUtensorMap mapC, const GemmArgs g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // align dynamic smem to 1024 B (SWIZZLE_128B atoms)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int b_tile_bytes = g.BN * kBK * 2;
  const int stage_bytes = kATileBytes + b_tile_bytes;
  uint8_t* stage_c = smem + (size_t)g.stages * stage_bytes;  // 2 x [128 rows][64 B] output slabs (SWIZZLE_64B)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(stage_c + kCSlabs * 8192);
  uint64_t* empty_bar = full_bar + g.stages;
  uint64_t* tfull_bar = empty_bar + g.stages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&mapA);
    tma_prefetch_desc(&mapB);
    if (g.tma_store) tma_prefetch_desc(&mapC);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < g.stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull_bar[i], 1);
      mbar_init(&tempty_bar[i], 256);
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const long total_tiles = (long)g.batch * g.splits * g.m_tiles * g.n_tiles;

  if (warp == 0) {
    // ===================== TMA producer (whole warp runs the control flow, one elected lane issues) ============
    {
      int s = 0;
      uint32_t ph = 0;
      for (long t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        const int n_t = (int)(t % g.n_tiles);
        long r = t / g.n_tiles;
        const int m_t = (int)(r % g.m_tiles);
        r /= g.m_tiles;
        const int sp = (int)(r % g.splits);
        const int bz = (int)(r / g.splits);
        const int m0 = m_t * kBM, n0 = n_t * g.BN;
        const int kc0 = sp * g.kper;
        const int kc1 = min(g.kchunks, kc0 + g.kper);
        // first output pixel of the tile: image cb0, row ch0, column cw0 (cw0 > 0 only for images wider than 128,
        // where a tile is a 128-pixel segment of one row)
        int cb0 = 0, ch0 = 0, cw0 = 0;
        if (g.conv == 1) {
          const int img = g.H * g.W;
          cb0 = m0 / img;
          ch0 = (m0 % img) / g.W;
          cw0 = m0 % g.W;
        }
        for (int kc = kc0; kc < kc1; ++kc) {
          mbar_wait(&empty_bar[s], ph ^ 1u);
          uint8_t* sA = smem + (size_t)s * stage_bytes;
          uint8_t* sB = sA + kATileBytes;
          if (g.debug & 8) {          // probe: no operand traffic at all (MMA + barrier rate on stale smem)
            if (elect_one()) mbar_arrive(&full_bar[s]);
          } else
          if (elect_one()) {
          mbar_expect_tx(&full_bar[s], (uint32_t)stage_bytes);
          if (g.conv == 2) {
            // 3x3 weight gradient: dW[tap][co][ci] = sum_p dY[p][co] * X[p + tap][ci].  A = dY (MN-major, 64 pixels of
            // K per chunk), B = the tap-shifted input pixels (MN-major; same 4-D box + out-of-bounds zero fill as the
            // forward's A operand, 64 pixels x 64 channels per N chunk); batch index = tap
            const int tap = bz, dy = tap / 3, dx = tap % 3;
            const int p0 = kc * kBK, img = g.H * g.W;
            const int b0 = p0 / img, h0 = (p0 % img) / g.W;
            tma_load_3d(sA, &mapA, &full_bar[s], m0, p0, 0);
            tma_load_3d(sA + 8192, &mapA, &full_bar[s], m0 + 64, p0, 0);
            for (int i = 0; i < g.BN / 64; ++i)
              tma_load_4d(sB + i * 8192, &mapB, &full_bar[s], n0 + 64 * i, dx - 1, h0 + dy - 1, b0);
          } else if (g.conv) {
            const int tap = kc / g.cin_chunks, cc = kc % g.cin_chunks;
            const int dy = tap / 3, dx = tap % 3;
            tma_load_4d(sA, &mapA, &full_bar[s], cc * kBK, g.cstride * cw0 + dx - g.cpad, g.cstride * ch0 + dy - g.cpad,
                        cb0);
            tma_load_2d(sB, &mapB, &full_bar[s], cc * kBK, tap * g.cout + n0);
          } else {
            const int ab = g.a_batched ? bz : 0, bb = g.b_batched ? bz : 0;
            if (!g.a_mn) {
              tma_load_3d(sA, &mapA, &full_bar[s], kc * kBK, m0, ab);
            } else {
              tma_load_3d(sA, &mapA, &full_bar[s], m0, kc * kBK, ab);
              tma_load_3d(sA + 8192, &mapA, &full_bar[s], m0 + 64, kc * kBK, ab);
            }
            if (!g.b_mn) {
              tma_load_3d(sB, &mapB, &full_bar[s], kc * kBK, n0, bb);
            } else {
              for (int i = 0; i < g.BN / 64; ++i)
                tma_load_3d(sB + i * 8192, &mapB, &full_bar[s], n0 + 64 * i, kc * kBK, bb);
            }
          }
          }  // elect_one
          __syncwarp();
          if (++s == g.stages) {
            s = 0;
            ph ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp runs the control flow, one elected lane issues) ==============
    {
      const uint32_t idesc = umma_idesc_bf16((uint32_t)g.BN, g.a_mn != 0, g.b_mn != 0);
      // descriptors of stage 0 / k-step 0; a later stage or k-step only moves the 14-bit start-address field
      // (all of shared memory is below 256 KiB, so the addition never carries out of the field)
      const uint32_t s0 = smem_u32(smem);
      const uint64_t dA0 = g.a_mn ? umma_desc(s0, 8192, 1024) : umma_desc(s0, 16, 1024);
      const uint64_t dB0 = g.b_mn ? umma_desc(s0 + kATileBytes, 8192, 1024) : umma_desc(s0 + kATileBytes, 16, 1024);
      const uint32_t a_step = g.a_mn ? (2048u >> 4) : (32u >> 4);
      const uint32_t b_step = g.b_mn ? (2048u >> 4) : (32u >> 4);
      const uint32_t stage_units = (uint32_t)stage_bytes >> 4;
      int s = 0, as = 0;
      uint32_t ph = 0, aph = 0;
      // (round 2, measured and removed: per-WARP output staging with 32x32 TMA stores instead of 128-thread slabs, no
      // CTA-level barrier in the slab loop — 65536x960x320 49.9 us vs 48.3 us, 65536x320x320 21.6 vs 20.1 us, r02 call 10)
      // (round 2, measured and removed: polling the NEXT stage's mbarrier before issuing the current stage's MMAs — with
      // try_wait 1.3-1.5x slower (it may suspend the thread), with the non-blocking test_wait 3-7 % slower, and even the
      // dormant branch cost 5-10 % in this loop; the issue loop itself, barriers only, is ~290 clk per k-chunk)
      for (long t = blockIdx.x; t < total_tiles; t += gridDim.x) {
        long r = t / g.n_tiles / g.m_tiles;
        const int sp = (int)(r % g.splits);
        const int kc0 = sp * g.kper;
        const int kc1 = min(g.kchunks, kc0 + g.kper);
        mbar_wait(&tempty_bar[as], aph ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)as * 256u;
        for (int kc = kc0; kc < kc1; ++kc) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t da = dA0 + (uint64_t)((uint32_t)s * stage_units);
            const uint64_t db = dB0 + (uint64_t)((uint32_t)s * stage_units);
            if (!(g.debug & 16)) {      // probe bit 16: no MMAs (TMA delivery rate alone)
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k)
              umma_bf16(d_tmem, da + (uint64_t)(k * a_step), db + (uint64_t)(k * b_step), idesc,
                        (kc > kc0 || k > 0) ? 1u : 0u);
            }
            umma_commit(&empty_bar[s]);  // frees the smem stage when these MMAs retire
          }
          __syncwarp();
          if (++s == g.stages) {
            s = 0;
            ph ^= 1u;
          }
        }
        if (elect_one()) umma_commit(&tfull_bar[as]);  // accumulator complete -> epilogue
        __syncwarp();
        as ^= 1;
        if (as == 0) aph ^= 1u;
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (256 threads: one accumulator row each, two column halves) ==============
    // warp (4 + 4*half + e) owns TMEM lanes [32e, 32e+32) and the 32-column slabs with (slab & 1) == half.
    const int ew = (warp - 4) & 3;   // == warp % 4 -> TMEM lane quadrant
    const int half = (warp - 4) >> 2;
    const int row = ew * 32 + lane;
    int as = 0;
    uint32_t aph = 0;
    uint32_t slab_ctr = 0;
    for (long t = blockIdx.x; t < total_tiles; t += gridDim.x) {
      const int n_t = (int)(t % g.n_tiles);
      long r = t / g.n_tiles;
      const int m_t = (int)(r % g.m_tiles);
      r /= g.m_tiles;
      const int bz = (int)(r / g.splits);
      const int m = m_t * kBM + row;
      const int n0 = n_t * g.BN;
      mbar_wait(&tfull_bar[as], aph);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (uint32_t)as * 256u + ((uint32_t)(ew * 32) << 16);
      const bool row_ok = m < g.M;
      const float* rg = (g.rowgroup && row_ok) ? g.rowgroup + (long long)(m / g.rows_per_group) * g.N : nullptr;
      const bf16* res = (g.residual && row_ok) ? g.residual + (long long)bz * g.res_bstride + (long long)m * g.ldr
                                               : nullptr;
      if (g.debug & 1) {
      } else if (g.tma_store && g.epi_plain && g.alpha == 1.f) {
        // ---- plain bf16 output (QKV projections, every dX GEMM) or bias only (FF / ViT linears): the general loop
        // below predicates its row-group / residual code instead of branching around it (~380 issued instructions per
        // 32-column slab, 60 % of them predicated off; a bias alone cost +10 us on 65536 x 320 x 320); this copy carries
        // only the (warp-uniformly branched) bias add.
        const bool lead_warp = (ew == 0);
        const uint32_t sw = ((uint32_t)row >> 1) & 3u;
        uint32_t v[32];
        int c = 32 * half;
        // residual (warp-uniform flag; rows past M read row M-1, their results are clipped by the TMA store): the 64 bytes a
        // thread needs for a slab are fetched ONE SLAB AHEAD
        const bool has_res = g.residual != nullptr;
        const bf16* resc = has_res ? g.residual + (long long)bz * g.res_bstride + (long long)(row_ok ? m : g.M - 1) * g.ldr
                                   : nullptr;
        uint4 rv[4];
        auto load_res = [&](int cc) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int n = n0 + cc + q * 8;
            rv[q] = (n + 8 <= g.N) ? *reinterpret_cast<const uint4*>(resc + n) : make_uint4(0, 0, 0, 0);
          }
        };
        if (c < g.BN && n0 + c < g.N) {
          __syncwarp();
          tmem_ld32(t_row + (uint32_t)c, v);
          if (has_res) load_res(c);
        }
        for (; c < g.BN && n0 + c < g.N; c += 64) {
          tmem_ld_wait();
          if (has_res) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float2 r0 = unpack_bf16(rv[q].x), r1 = unpack_bf16(rv[q].y), r2 = unpack_bf16(rv[q].z),
                           r3 = unpack_bf16(rv[q].w);
              v[8 * q + 0] = __float_as_uint(__uint_as_float(v[8 * q + 0]) + r0.x);
              v[8 * q + 1] = __float_as_uint(__uint_as_float(v[8 * q + 1]) + r0.y);
              v[8 * q + 2] = __float_as_uint(__uint_as_float(v[8 * q + 2]) + r1.x);
              v[8 * q + 3] = __float_as_uint(__uint_as_float(v[8 * q + 3]) + r1.y);
              v[8 * q + 4] = __float_as_uint(__uint_as_float(v[8 * q + 4]) + r2.x);
              v[8 * q + 5] = __float_as_uint(__uint_as_float(v[8 * q + 5]) + r2.y);
              v[8 * q + 6] = __float_as_uint(__uint_as_float(v[8 * q + 6]) + r3.x);
              v[8 * q + 7] = __float_as_uint(__uint_as_float(v[8 * q + 7]) + r3.y);
            }
          }
          if (g.rowgroup) {   // warp-uniform flag: per-image time-embedding row of ResnetBlock2D.conv1 (fp32 [M / rpg][N])
            const float* rgr = g.rowgroup + (long long)((row_ok ? m : g.M - 1) / g.rows_per_group) * g.N;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const int n = n0 + c + q * 4;
              if (n + 4 <= g.N) {
                const float4 b = *reinterpret_cast<const float4*>(rgr + n);
                v[4 * q + 0] = __float_as_uint(__uint_as_float(v[4 * q + 0]) + b.x);
                v[4 * q + 1] = __float_as_uint(__uint_as_float(v[4 * q + 1]) + b.y);
                v[4 * q + 2] = __float_as_uint(__uint_as_float(v[4 * q + 2]) + b.z);
                v[4 * q + 3] = __float_as_uint(__uint_as_float(v[4 * q + 3]) + b.w);
              }
            }
          }
          uint32_t w[16];
          if (g.bias) {   // warp-uniform: Linear / conv bias (fp32, same 32 values for every row: L1 broadcast loads)
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const int n = n0 + c + q * 4;
              float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
              if (n + 4 <= g.N) b = *reinterpret_cast<const float4*>(g.bias + n);
              w[2 * q] = pack_bf16(__uint_as_float(v[4 * q]) + b.x, __uint_as_float(v[4 * q + 1]) + b.y);
              w[2 * q + 1] = pack_bf16(__uint_as_float(v[4 * q + 2]) + b.z, __uint_as_float(v[4 * q + 3]) + b.w);
            }
          } else {
#pragma unroll
            for (int q = 0; q < 16; ++q) w[q] = pack_bf16(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1]));
          }
          const int cn = c + 64;
          if (cn < g.BN && n0 + cn < g.N) {
            __syncwarp();
            tmem_ld32(t_row + (uint32_t)cn, v);
            if (has_res) load_res(cn);
          }
          uint8_t* slab = stage_c + (half + 2 * (slab_ctr & 1)) * 8192;
          if (lead_warp) {
            if (elect_one()) tma_store_wait_read<1>();  // the store that last read this slab has drained
          }
          if (half == 0) asm volatile("bar.sync 3, 128;" ::: "memory");
          else asm volatile("bar.sync 5, 128;" ::: "memory");
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(slab + row * 64 + ((((uint32_t)q) ^ sw) << 4)) =
                make_uint4(w[q * 4], w[q * 4 + 1], w[q * 4 + 2], w[q * 4 + 3]);
          fence_proxy_async_smem();
          if (half == 0) asm volatile("bar.sync 4, 128;" ::: "memory");
          else asm volatile("bar.sync 6, 128;" ::: "memory");
          if (lead_warp) {
            if (elect_one()) {
              tma_store_3d(&mapC, slab, n0 + c, m_t * kBM, bz);
              tma_store_commit();
            }
          }
          ++slab_ctr;
        }
      } else if (g.tma_store) {
        // ---- bf16 output: registers -> swizzled smem slab -> TMA store (full-line coalesced writes) ----
        const bool lead_warp = (ew == 0);   // warp-uniform; its elected lane owns this half's TMA-store bulk groups
        const uint32_t sw = ((uint32_t)row >> 1) & 3u;
        uint32_t v[32];
        int c = 32 * half;
        const bool any = (c < g.BN && n0 + c < g.N);
        if (any) {
          __syncwarp();
          tmem_ld32(t_row + (uint32_t)c, v);
        }
        for (; c < g.BN && n0 + c < g.N; c += 64) {
          tmem_ld_wait();
          uint32_t w[16];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int n = n0 + c + q * 8;
            float f[8];
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) f[jj] = __uint_as_float(v[q * 8 + jj]) * g.alpha;
            if (n + 8 <= g.N) {
              if (g.bias) {
                const float4 b0 = *reinterpret_cast<const float4*>(g.bias + n);
                const float4 b1 = *reinterpret_cast<const float4*>(g.bias + n + 4);
                f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
                f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
              }
              if (rg) {
                const float4 b0 = *reinterpret_cast<const float4*>(rg + n);
                const float4 b1 = *reinterpret_cast<const float4*>(rg + n + 4);
                f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
                f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
              }
              if (res) {   // (only with a row-group addend or alpha != 1: every other residual goes through the lean loop)
                const uint4 rvq = *reinterpret_cast<const uint4*>(res + n);
                const float2 r0 = unpack_bf16(rvq.x), r1 = unpack_bf16(rvq.y), r2 = unpack_bf16(rvq.z),
                             r3 = unpack_bf16(rvq.w);
                f[0] += r0.x; f[1] += r0.y; f[2] += r1.x; f[3] += r1.y;
                f[4] += r2.x; f[5] += r2.y; f[6] += r3.x; f[7] += r3.y;
              }
            }
            w[q * 4 + 0] = pack_bf16(f[0], f[1]);
            w[q * 4 + 1] = pack_bf16(f[2], f[3]);
            w[q * 4 + 2] = pack_bf16(f[4], f[5]);
            w[q * 4 + 3] = pack_bf16(f[6], f[7]);
          }
          // prefetch the next slab of this half while the current one is staged and stored
          const int cn = c + 64;
          if (cn < g.BN && n0 + cn < g.N) {
            __syncwarp();
            tmem_ld32(t_row + (uint32_t)cn, v);
          }
          if (g.debug & 4) continue;
          // this half cycles through staging slabs {half, half + 2}
          uint8_t* slab = stage_c + (half + 2 * (slab_ctr & 1)) * 8192;
          if (lead_warp) {
            if (elect_one()) tma_store_wait_read<1>();  // the store that last read this slab has drained
          }
          if (half == 0) asm volatile("bar.sync 3, 128;" ::: "memory");
          else asm volatile("bar.sync 5, 128;" ::: "memory");
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(slab + row * 64 + ((((uint32_t)q) ^ sw) << 4)) =
                make_uint4(w[q * 4], w[q * 4 + 1], w[q * 4 + 2], w[q * 4 + 3]);
          fence_proxy_async_smem();
          if (half == 0) asm volatile("bar.sync 4, 128;" ::: "memory");
          else asm volatile("bar.sync 6, 128;" ::: "memory");
          if (lead_warp) {
            if (elect_one()) {
              tma_store_3d(&mapC, slab, n0 + c, m_t * kBM, bz);
              tma_store_commit();
            }
          }
          ++slab_ctr;
        }
      } else
      for (int c = 32 * half; c < g.BN; c += 64) {
        uint32_t v[32];
        __syncwarp();
        tmem_ld32(t_row + (uint32_t)c, v);
        tmem_ld_wait();
        if (row_ok) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int n = n0 + c + q * 8;
          if (n >= g.N) break;
          float f[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = __uint_as_float(v[q * 8 + j]) * g.alpha;
          const bool full8 = g.epi_vec && (n + 8 <= g.N);
          if (full8) {
            if (g.bias) {
              const float4 b0 = *reinterpret_cast<const float4*>(g.bias + n);
              const float4 b1 = *reinterpret_cast<const float4*>(g.bias + n + 4);
              f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
              f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
            }
            if (rg) {
              const float4 b0 = *reinterpret_cast<const float4*>(rg + n);
              const float4 b1 = *reinterpret_cast<const float4*>(rg + n + 4);
              f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
              f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
            }
            if (res) {
              const uint4 rv = *reinterpret_cast<const uint4*>(res + n);
              const float2 r0 = unpack_bf16(rv.x), r1 = unpack_bf16(rv.y), r2 = unpack_bf16(rv.z),
                           r3 = unpack_bf16(rv.w);
              f[0] += r0.x; f[1] += r0.y; f[2] += r1.x; f[3] += r1.y;
              f[4] += r2.x; f[5] += r2.y; f[6] += r3.x; f[7] += r3.y;
            }
            if (g.out_mode == 0) {
              bf16* o = reinterpret_cast<bf16*>(g.out) + (long long)bz * g.out_bstride + (long long)m * g.ldo + n;
              uint4 ov;
              ov.x = pack_bf16(f[0], f[1]); ov.y = pack_bf16(f[2], f[3]);
              ov.z = pack_bf16(f[4], f[5]); ov.w = pack_bf16(f[6], f[7]);
              *reinterpret_cast<uint4*>(o) = ov;
            } else if (g.out_mode == 1) {
              float* o = reinterpret_cast<float*>(g.out) + (long long)bz * g.out_bstride + (long long)m * g.ldo + n;
              *reinterpret_cast<float4*>(o) = make_float4(f[0], f[1], f[2], f[3]);
              *reinterpret_cast<float4*>(o + 4) = make_float4(f[4], f[5], f[6], f[7]);
            } else {
              float* o = reinterpret_cast<float*>(g.out) + (long long)bz * g.out_bstride + (long long)m * g.ldo + n;
#pragma unroll
              for (int j = 0; j < 8; ++j) atomicAdd(o + j, f[j]);
            }
          } else {
            for (int j = 0; j < 8 && n + j < g.N; ++j) {
              float x = f[j];
              if (g.bias) x += g.bias[n + j];
              if (rg) x += rg[n + j];
              if (res) x += __bfloat162float(res[n + j]);
              const long long off = (long long)bz * g.out_bstride + (long long)m * g.ldo + n + j;
              if (g.out_mode == 0) reinterpret_cast<bf16*>(g.out)[off] = __float2bfloat16(x);
              else if (g.out_mode == 1) reinterpret_cast<float*>(g.out)[off] = x;
              else atomicAdd(reinterpret_cast<float*>(g.out) + off, x);
            }
          }
        }
        }  // row_ok
      }
      tc_fence_before();
      mbar_arrive(&tempty_bar[as]);
      as ^= 1;
      if (as == 0) aph ^= 1u;
    }
    if (g.tma_store && (warp == 4 || warp == 8)) {
      if (elect_one()) tma_store_wait_all();  // smem must outlive the stores (same lane that committed them)
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
static int g_num_sms = 0;
static int num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}

// Tile-width choice by a cost model FITTED to measurements (tools/sweep_r2.py gemm: every GEMM/conv signature of the
// pre-training step timed at every BN on a B200, profiles/r02_gemm_bn_sweep.md; rms log-error of the fit 9.5 %).
// In nominal cycles per CTA:
//   mainloop per 64-deep k-chunk  = 505 + 0.47 * BN   (operand delivery dominates: the cost is almost flat in BN, so the
//                                                      widest tile that does not add a round of the persistent grid wins)
//   epilogue per tile             = 2060 + 21.6 * BN * (1 + 1.07 * [residual]) * (6 if fp32 atomics)
//   tile                          = max(mainloop, epilogue)   (the epilogue of tile i overlaps the mainloop of i+1)
//   kernel                        = ceil(tiles / SMs) * tile + epilogue
// Choosing BN with this model costs 39.1 ms/step over the 116 signatures, against 38.8 ms for the per-signature best and
// 44.4 ms for the round-1 model (max(2*BN, 128+BN) per chunk), which preferred tiles that were too narrow.
static int pick_bn(int N, long m_tiles_x_batch, bool b_mn, int force_bn, int kchunks_per_tile = 16,
                   bool residual = false, bool atomic = false, double* cost_out = nullptr) {
  if (force_bn > 0) return force_bn;
  const int step = b_mn ? 64 : 32;
  int best = 0;
  double best_cost = 1e30;
  const double sms = (double)num_sms();
  for (int bn = 256; bn >= 64; bn -= step) {
    const int tiles_n = cdiv(N, bn);
    const double tiles = (double)tiles_n * (double)m_tiles_x_batch;
    const double mainloop = kchunks_per_tile * (505.0 + 0.47 * bn);
    const double epilogue = 2060.0 + 21.6 * bn * (residual ? 2.07 : 1.0) * (atomic ? 6.0 : 1.0);
    const double tile = mainloop > epilogue ? mainloop : epilogue;
    const double rounds = (double)((long)((tiles + sms - 1) / sms));
    const double cost = rounds * tile + epilogue;
    if (cost < best_cost - 1e-6) {
      best_cost = cost;
      best = bn;
    }
  }
  if (cost_out) *cost_out = best_cost;
  return best;
}

// Split-K factor of an fp32-accumulating GEMM (weight gradients: small M x N, very long K) by the same cost model: the
// factor that minimises rounds x max(mainloop, atomic epilogue) + epilogue.  (Round 2: "fill the machine about twice"
// from 128 x 128 tile counts gave e.g. 13 splits x 16 tiles = 208 CTAs for the level-0 QKV weight gradient — 1.4 rounds of
// the 148-CTA persistent grid; 9 splits = 144 CTAs do the same work in one.)
static int auto_splits(int N, long m_tiles_x_batch, bool b_mn, int kchunks) {
  int best = 1;
  double best_cost = 1e30;
  const int smax = kchunks < 64 ? kchunks : 64;
  for (int sp = 1; sp <= smax; ++sp) {
    const int kper = cdiv(kchunks, sp);
    if (cdiv(kchunks, kper) != sp) continue;          // same kper as a smaller factor
    double c = 0;
    pick_bn(N, m_tiles_x_batch * sp, b_mn, 0, kper, false, true, &c);
    if (c < best_cost - 1e-6) {
      best_cost = c;
      best = sp;
    }
  }
  return best;
}

static int launch_gemm(const CUtensorMap& mA, const CUtensorMap& mB, GemmArgs& g, cudaStream_t stream) {
  // output map for the TMA-store epilogue: bf16 [batch][M][N], box 32 cols x 128 rows, SWIZZLE_64B
  CUtensorMap mC;
  memset(&mC, 0, sizeof(mC));
  g.tma_store = 0;
  {
    const char* d = getenv("E4T_GEMM_DEBUG");
    g.debug = d ? atoi(d) : 0;
    const char* p = getenv("E4T_GEMM_EPI_PLAIN");   // default ON (bit-identical on all 40 step signatures, r02 sweep)
    g.epi_plain = p ? atoi(p) : 1;
  }
  static int use_tma_store = -1;
  if (use_tma_store < 0) {
    const char* e = getenv("E4T_GEMM_TMA_STORE");
    use_tma_store = (e && e[0] == '0') ? 0 : 1;
  }
  // Epilogue alignment (include/e4t_b200.h).  Bias and row-group rows are read as float4 at multiples of 8 columns on
  // every path, so their base pointers must be 16-byte aligned.  The output, residual and row-group row strides only
  // choose the path: every 16-byte access of the per-thread loop is aligned (epi_vec), or that loop goes scalar.
  E4T_CHECK(((uintptr_t)g.bias % 16) == 0 && ((uintptr_t)g.rowgroup % 16) == 0,
            "e4t_gemm: bias and rowgroup must be 16-byte aligned");
  const int out_el = g.out_mode == 0 ? 8 : 4;  // output elements per 16 bytes
  const bool out_vec = g.out_mode == 2 || (((uintptr_t)g.out % 16) == 0 && (g.ldo % out_el) == 0 &&
                                           (g.batch == 1 || (g.out_bstride % out_el) == 0));
  const bool res_vec = !g.residual || (((uintptr_t)g.residual % 16) == 0 && (g.ldr % 8) == 0 &&
                                       (g.batch == 1 || (g.res_bstride % 8) == 0));
  const bool rg_vec = !g.rowgroup || (g.N % 4) == 0;
  g.epi_vec = out_vec && res_vec && rg_vec;
  if (use_tma_store && g.out_mode == 0 && (g.N % 8) == 0 && (g.ldo % 8) == 0 && ((uintptr_t)g.out % 16) == 0 &&
      (g.batch == 1 || (g.out_bstride % 8) == 0) && res_vec) {
    uint64_t dims[3] = {(uint64_t)g.N, (uint64_t)g.M, (uint64_t)g.batch};
    uint64_t str[2] = {(uint64_t)g.ldo * 2, (uint64_t)(g.batch > 1 ? g.out_bstride : (long long)g.M * g.ldo) * 2};
    uint32_t box[3] = {32, kBM, 1};
    if (int e = e4t_tmap_encode(&mC, g.out, 3, dims, str, box, 2, 64)) return e;
    g.tma_store = 1;
  }
  const int stage_bytes = kATileBytes + g.BN * kBK * 2;
  int stages = (192 * 1024) / stage_bytes;
  if (stages > 8) stages = 8;
  if (stages > g.kper) stages = g.kper < 2 ? 2 : g.kper;
  g.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + kCSlabs * 8192 + (2 * stages + 4) * sizeof(uint64_t) + 16 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    E4T_CUDA(cudaFuncSetAttribute(e4t_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  const long total = (long)g.batch * g.splits * g.m_tiles * g.n_tiles;
  int grid = (int)(total < num_sms() ? total : num_sms());
  if (grid < 1) return 0;
  e4t_gemm_kernel<<<grid, kThreads, smem, stream>>>(mA, mB, mC, g);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}

extern "C" int e4t_gemm_bf16(const void* A, const void* B, void* out, int M, int N, int K, int batch, int a_mn,
                             int b_mn, long long lda, long long ldb, long long a_bstride, long long b_bstride,
                             int out_mode, long long ldo, long long out_bstride, const float* bias,
                             const float* rowgroup, int rows_per_group, const void* residual, long long ldr,
                             long long res_bstride, float alpha, int splits, int force_bn, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  E4T_CHECK(M > 0 && N > 0 && K > 0 && batch > 0, "e4t_gemm_bf16: bad dims M=%d N=%d K=%d batch=%d", M, N, K, batch);
  E4T_CHECK((lda % 8) == 0 && (ldb % 8) == 0, "e4t_gemm_bf16: leading strides must be multiples of 8 elements");
  E4T_CHECK(((uintptr_t)A % 16) == 0 && ((uintptr_t)B % 16) == 0, "e4t_gemm_bf16: operands must be 16-byte aligned");
  E4T_CHECK(out_mode >= 0 && out_mode <= 2, "e4t_gemm_bf16: bad out_mode");
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = M; g.N = N; g.K = K; g.batch = batch;
  g.a_mn = a_mn; g.b_mn = b_mn;
  g.a_batched = (a_bstride != 0); g.b_batched = (b_bstride != 0);
  g.m_tiles = cdiv(M, kBM);
  g.kchunks = cdiv(K, kBK);
  if (splits == 0 && out_mode == 2 && force_bn <= 0) splits = auto_splits(N, (long)g.m_tiles * batch, b_mn != 0, g.kchunks);
  if (splits < 1) splits = 1;
  if (splits > g.kchunks) splits = g.kchunks;
  g.kper = cdiv(g.kchunks, splits);
  g.splits = cdiv(g.kchunks, g.kper);  // no empty split
  g.BN = pick_bn(N, (long)g.m_tiles * batch * g.splits, b_mn != 0, force_bn, g.kper, residual != nullptr, out_mode == 2);
  E4T_CHECK(g.BN >= 32 && g.BN <= 256 && (g.BN % (b_mn ? 64 : 32)) == 0, "e4t_gemm_bf16: bad BN %d", g.BN);
  g.n_tiles = cdiv(N, g.BN);
  E4T_CHECK(g.splits == 1 || out_mode == 2, "e4t_gemm_bf16: split-K requires atomic fp32 output");
  // every split would add them again
  E4T_CHECK(g.splits == 1 || (!bias && !rowgroup && !residual), "e4t_gemm_bf16: split-K takes no bias/rowgroup/residual");
  g.out = out; g.out_mode = out_mode; g.ldo = ldo; g.out_bstride = out_bstride;
  g.bias = bias; g.rowgroup = rowgroup; g.rows_per_group = rows_per_group > 0 ? rows_per_group : 1;
  g.residual = (const bf16*)residual; g.ldr = ldr; g.res_bstride = res_bstride;
  g.alpha = alpha;

  CUtensorMap mA, mB;
  {
    const uint64_t nb = g.a_batched ? (uint64_t)batch : 1;
    const uint64_t bs = g.a_batched ? (uint64_t)a_bstride : (uint64_t)lda * (a_mn ? K : M);
    if (!a_mn) {
      uint64_t dims[3] = {(uint64_t)K, (uint64_t)M, nb};
      uint64_t str[2] = {(uint64_t)lda * 2, bs * 2};
      uint32_t box[3] = {kBK, kBM, 1};
      if (int e = e4t_tmap_encode(&mA, A, 3, dims, str, box, 2)) return e;
    } else {
      uint64_t dims[3] = {(uint64_t)M, (uint64_t)K, nb};
      uint64_t str[2] = {(uint64_t)lda * 2, bs * 2};
      uint32_t box[3] = {64, kBK, 1};
      if (int e = e4t_tmap_encode(&mA, A, 3, dims, str, box, 2)) return e;
    }
  }
  {
    const uint64_t nb = g.b_batched ? (uint64_t)batch : 1;
    const uint64_t bs = g.b_batched ? (uint64_t)b_bstride : (uint64_t)ldb * (b_mn ? K : N);
    if (!b_mn) {
      uint64_t dims[3] = {(uint64_t)K, (uint64_t)N, nb};
      uint64_t str[2] = {(uint64_t)ldb * 2, bs * 2};
      uint32_t box[3] = {kBK, (uint32_t)g.BN, 1};
      if (int e = e4t_tmap_encode(&mB, B, 3, dims, str, box, 2)) return e;
    } else {
      uint64_t dims[3] = {(uint64_t)N, (uint64_t)K, nb};
      uint64_t str[2] = {(uint64_t)ldb * 2, bs * 2};
      uint32_t box[3] = {64, kBK, 1};
      if (int e = e4t_tmap_encode(&mB, B, 3, dims, str, box, 2)) return e;
    }
  }
  return launch_gemm(mA, mB, g, stream);
}

// x: NHWC bf16 [B][Hin][Win][Cin];  w: bf16 [9][Cout][Cin] (tap = ky*3+kx);  out: [B*H*W][Cout] (NHWC), H = Hin/stride.
// pad 1.  bias fp32 [Cout]; rowgroup fp32 [B][Cout] (time-embedding projection) ; residual bf16 NHWC.
// stride 2 (diffusers Downsample2D): the A-operand tensor map walks the input with element strides (1,2,2,1), so the
// tile of 128 OUTPUT pixels is gathered directly from every other input pixel — no stride-1 result is computed and
// thrown away (round 1 did exactly that: 4x the FLOPs on the three downsampling convolutions).
// Output widths above 128 (the VAE at 256 and 512 pixels) must be multiples of 128: each 128-row M tile is then a
// 128-pixel segment of one image row, and the producer offsets the A-operand box by the segment's first column.
// pad 0 (stride 2 only): diffusers' VAE Downsample2D, F.pad(x, (0,1,0,1)) then a pad-0 conv; the bottom/right zero
// row and column come from the TMA out-of-bounds fill.
static int conv3x3_impl(const void* x, const void* w, void* out, int B, int Hin, int Win, int Cin, int Cout, int stride,
                        int pad, int out_mode, const float* bias, const float* rowgroup, const void* residual,
                        int force_bn, cudaStream_t stream) {
  E4T_CHECK(Cin % 64 == 0, "e4t_conv3x3: Cin must be a multiple of 64 (got %d)", Cin);
  E4T_CHECK(stride == 1 || (stride == 2 && Hin % 2 == 0 && Win % 2 == 0), "e4t_conv3x3: bad stride/size");
  E4T_CHECK(pad == 1 || (pad == 0 && stride == 2), "e4t_conv3x3: pad must be 1, or 0 with stride 2 (got %d)", pad);
  const int H = Hin / stride, W = Win / stride;
  E4T_CHECK((W <= 128 && (128 % W) == 0) || (W % 128) == 0,
            "e4t_conv3x3: output width must divide 128 or be a multiple of 128 (got %d)", W);
  E4T_CHECK(out_mode == 0 || out_mode == 1, "e4t_conv3x3: bad out_mode");
  const int img = H * W;
  int BH, BB;
  if (W >= 128) {
    BB = 1;
    BH = 1;
  } else if (img >= 128) {
    BB = 1;
    BH = 128 / W;
    E4T_CHECK(H % BH == 0, "e4t_conv3x3: H=%d not a multiple of tile height %d", H, BH);
  } else {
    E4T_CHECK(128 % img == 0, "e4t_conv3x3: H*W must divide 128");
    BB = 128 / img;
    BH = H;
  }
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = B * img; g.N = Cout; g.K = Cin; g.batch = 1;
  g.conv = 1; g.H = H; g.W = W; g.BH = BH; g.BB = BB; g.cin_chunks = Cin / 64; g.cout = Cout; g.cstride = stride;
  g.cpad = pad;
  g.m_tiles = cdiv(g.M, kBM);
  g.kchunks = 9 * g.cin_chunks;
  g.kper = g.kchunks; g.splits = 1;
  g.BN = pick_bn(Cout, g.m_tiles, false, force_bn, g.kchunks, residual != nullptr, false);
  E4T_CHECK(g.BN >= 32 && g.BN <= 256 && (g.BN % 32) == 0, "e4t_conv3x3: bad BN %d", g.BN);
  g.n_tiles = cdiv(Cout, g.BN);
  g.out = out; g.out_mode = out_mode; g.ldo = Cout; g.out_bstride = 0;
  g.bias = bias; g.rowgroup = rowgroup; g.rows_per_group = img;
  g.residual = (const bf16*)residual; g.ldr = Cout; g.res_bstride = 0;
  g.alpha = 1.f;
  CUtensorMap mA, mB;
  {
    uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)Win, (uint64_t)Hin, (uint64_t)B};
    uint64_t str[3] = {(uint64_t)Cin * 2, (uint64_t)Win * Cin * 2, (uint64_t)Hin * Win * Cin * 2};
    // (stride 2 at a 128-wide tile: a 256-element box with element stride 2, the largest box TMA takes)
    uint32_t box[4] = {kBK, (uint32_t)((W < 128 ? W : 128) * stride), (uint32_t)(BH * stride), (uint32_t)BB};
    uint32_t es[4] = {1, (uint32_t)stride, (uint32_t)stride, 1};
    if (int e = e4t_tmap_encode(&mA, x, 4, dims, str, box, 2, 128, stride == 1 ? nullptr : es)) return e;
  }
  {
    uint64_t dims[2] = {(uint64_t)Cin, (uint64_t)9 * Cout};
    uint64_t str[1] = {(uint64_t)Cin * 2};
    uint32_t box[2] = {kBK, (uint32_t)g.BN};
    if (int e = e4t_tmap_encode(&mB, w, 2, dims, str, box, 2)) return e;
  }
  return launch_gemm(mA, mB, g, stream);
}

extern "C" int e4t_conv3x3_bf16(const void* x, const void* w, void* out, int B, int H, int W, int Cin, int Cout,
                                int out_mode, const float* bias, const float* rowgroup, const void* residual,
                                int force_bn, void* stream_) {
  return conv3x3_impl(x, w, out, B, H, W, Cin, Cout, 1, 1, out_mode, bias, rowgroup, residual, force_bn,
                      (cudaStream_t)stream_);
}

// General forward 3x3 convolution (bf16 output): stride 1 or 2, top/left padding 1 or 0 (0 with stride 2 only), bias
// and residual in the epilogue; output widths that divide 128 or are multiples of 128.  x [B][H][W][Cin] ->
// out [B][H/stride][W/stride][Cout].
extern "C" int e4t_conv3x3_ex(const void* x, const void* w, void* out, int B, int H, int W, int Cin, int Cout,
                              int stride, int pad, const float* bias, const void* residual, int force_bn,
                              void* stream_) {
  return conv3x3_impl(x, w, out, B, H, W, Cin, Cout, stride, pad, 0, bias, nullptr, residual, force_bn,
                      (cudaStream_t)stream_);
}

// 3x3 / stride 2 / pad 1 (diffusers Downsample2D.conv, e4t/models/unet_2d_blocks.py:801-808): x [B][H][W][Cin] ->
// out [B][H/2][W/2][Cout].
extern "C" int e4t_conv3x3_s2_bf16(const void* x, const void* w, void* out, int B, int H, int W, int Cin, int Cout,
                                   const float* bias, int force_bn, void* stream_) {
  return conv3x3_impl(x, w, out, B, H, W, Cin, Cout, 2, 1, 0, bias, nullptr, nullptr, force_bn, (cudaStream_t)stream_);
}

// 3x3 / stride 1 / pad 1 weight gradient: dw9[tap][co][ci] += sum_{b,y,x} dy[b][y][x][co] * x[b][y+ky-1][x+kx-1][ci]
// (tap = ky*3+kx; fp32 atomic accumulation, split-K over the pixels).  x NHWC bf16 [B][H][W][Cin], dy [B][H][W][Cout].
// Replaces autograd's conv2d weight gradient behind every ResnetBlock2D / Upsample2D / Downsample2D conv when the base
// UNet is trainable (tuning_e4t.py:139-146).  Cin, Cout % 64 == 0; W | 64; H*W % 64 == 0.
extern "C" int e4t_conv3x3_wgrad(const void* x, const void* dy, float* dw9, int B, int H, int W, int Cin, int Cout,
                                 void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  E4T_CHECK(Cin % 64 == 0 && Cout % 64 == 0, "e4t_conv3x3_wgrad: Cin, Cout must be multiples of 64 (%d, %d)", Cin, Cout);
  E4T_CHECK(W <= 64 && (64 % W) == 0 && (H * W) % 64 == 0 && H % (64 / W) == 0,
            "e4t_conv3x3_wgrad: unsupported image %dx%d (W | 64, H*W %% 64 == 0)", H, W);
  const long long pixels = (long long)B * H * W;
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = Cout; g.N = Cin; g.K = (int)pixels; g.batch = 9;
  g.a_mn = 1; g.b_mn = 1; g.a_batched = 0; g.b_batched = 1;
  g.conv = 2; g.H = H; g.W = W; g.cout = Cout; g.cstride = 1;
  g.m_tiles = cdiv(Cout, kBM);
  g.kchunks = (int)(pixels / kBK);
  // enough K-splits to fill the machine about twice: tiles = 9 taps x m_tiles x n_tiles x splits
  const int base_tiles = 9 * g.m_tiles * cdiv(Cin, 256);
  int splits = cdiv(2 * num_sms(), base_tiles);
  if (splits < 1) splits = 1;
  if (splits > g.kchunks) splits = g.kchunks;
  g.kper = cdiv(g.kchunks, splits);
  g.splits = cdiv(g.kchunks, g.kper);
  g.BN = Cin >= 256 ? 256 : (Cin >= 192 ? 192 : (Cin >= 128 ? 128 : 64));
  g.n_tiles = cdiv(Cin, g.BN);
  g.out = dw9; g.out_mode = 2; g.ldo = Cin; g.out_bstride = (long long)Cout * Cin;
  g.rows_per_group = 1; g.alpha = 1.f;
  CUtensorMap mA, mB;
  {
    uint64_t dims[3] = {(uint64_t)Cout, (uint64_t)pixels, 1};
    uint64_t str[2] = {(uint64_t)Cout * 2, (uint64_t)pixels * Cout * 2};
    uint32_t box[3] = {64, kBK, 1};
    if (int e = e4t_tmap_encode(&mA, dy, 3, dims, str, box, 2)) return e;
  }
  {
    uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)B};
    uint64_t str[3] = {(uint64_t)Cin * 2, (uint64_t)W * Cin * 2, (uint64_t)H * W * Cin * 2};
    uint32_t box[4] = {64, (uint32_t)W, (uint32_t)(64 / W), 1};
    if (int e = e4t_tmap_encode(&mB, x, 4, dims, str, box, 2)) return e;
  }
  return launch_gemm(mA, mB, g, stream);
}
