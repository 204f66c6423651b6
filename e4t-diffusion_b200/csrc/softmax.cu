// e4t_b200 — row softmax of an fp32 score matrix into bf16 probabilities: the middle launch of the VAE mid-block
// AttentionBlock (single head, head dim = C = 512, 1024-16384 tokens), whose core runs as
//   S = alpha * Q K^T (e4t_gemm_bf16, fp32 out)  ->  P = softmax_rows(S)  ->  O = P V (e4t_gemm_bf16, V MN-major).
// One CTA per row.  Pass 1 keeps a running (max, sum of exp) per thread over float4 loads and merges them across the
// CTA; pass 2 re-reads the row (64 KB at M = 16384, still in L2) and writes exp(s - max) / sum as bf16.
#include "common.cuh"

static constexpr int kSmThreads = 256;

__global__ void __launch_bounds__(kSmThreads)
softmax_rows_kernel(const float* __restrict__ S, bf16* __restrict__ P, int M, long long ld) {
  const float* s = S + (long long)blockIdx.x * ld;
  bf16* p = P + (long long)blockIdx.x * ld;
  __shared__ float red_m[kSmThreads / 32], red_s[kSmThreads / 32];
  const int n4 = M / 4;
  float mx = -INFINITY, sm = 0.f;
  for (int i = threadIdx.x; i < n4; i += kSmThreads) {
    const float4 v = reinterpret_cast<const float4*>(s)[i];
    const float m4 = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));
    if (m4 > mx) {
      sm *= __expf(mx - m4);
      mx = m4;
    }
    // (while every value seen is -inf, exp(-inf - -inf) would make the sum NaN for good)
    if (mx != -INFINITY) sm += __expf(v.x - mx) + __expf(v.y - mx) + __expf(v.z - mx) + __expf(v.w - mx);
  }
  // merge (max, sum) pairs: warp, then CTA
  float wm = warp_max(mx);
  float ws = warp_sum(mx == -INFINITY ? 0.f : sm * __expf(mx - wm));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    red_m[warp] = wm;
    red_s[warp] = ws;
  }
  __syncthreads();
  float rm = -INFINITY;
#pragma unroll
  for (int w = 0; w < kSmThreads / 32; ++w) rm = fmaxf(rm, red_m[w]);
  float rs = 0.f;
#pragma unroll
  for (int w = 0; w < kSmThreads / 32; ++w)
    if (red_m[w] != -INFINITY) rs += red_s[w] * __expf(red_m[w] - rm);
  const float inv = 1.f / rs;
  for (int i = threadIdx.x; i < n4; i += kSmThreads) {
    const float4 v = reinterpret_cast<const float4*>(s)[i];
    uint2 o;
    o.x = pack_bf16(__expf(v.x - rm) * inv, __expf(v.y - rm) * inv);
    o.y = pack_bf16(__expf(v.z - rm) * inv, __expf(v.w - rm) * inv);
    reinterpret_cast<uint2*>(p)[i] = o;
  }
}

extern "C" int e4t_softmax_rows(const float* S, void* P, long long rows, int M, long long ld, void* stream_) {
  E4T_CHECK(rows > 0 && rows <= 0x7fffffffLL && M > 0, "e4t_softmax_rows: bad dims rows=%lld M=%d", rows, M);
  E4T_CHECK(M % 4 == 0 && ld % 4 == 0 && ld >= M, "e4t_softmax_rows: M and ld must be multiples of 4, ld >= M");
  E4T_CHECK(((uintptr_t)S % 16) == 0 && ((uintptr_t)P % 8) == 0, "e4t_softmax_rows: misaligned S or P");
  softmax_rows_kernel<<<(unsigned)rows, kSmThreads, 0, (cudaStream_t)stream_>>>(S, (bf16*)P, M, ld);
  E4T_COUNT_LAUNCH();
  E4T_LAUNCH_CHECK();
  return 0;
}
