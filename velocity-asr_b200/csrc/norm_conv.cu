// norm_conv.cu — LayerNorm and the SSM block prologue (LayerNorm -> causal depthwise conv).
//
// Reference: F.layer_norm (eps 1e-5, biased variance) at model.py:200,224, ssm.py:408,423,504,
// attention.py:306-307; depthwise Conv1d(k, padding=k-1)[..., :L] at ssm.py:411-414.
// Both are streaming, HBM-bound kernels: one warp owns one token (C <= 1024 channels held in
// registers), rows are read and written once with fully coalesced 128-byte warp accesses.
#include "common.cuh"
#include "kernels.cuh"

namespace vasr {

namespace {

constexpr int LN_MAX_PER_LANE = 8;  // C <= 256 ... the model uses 192 (6 per lane)

// normalises one row held as v[i] = x[lane + 32*i]; returns through v.
template <int PER>
__device__ __forceinline__ void warp_layer_norm(float (&v)[PER], int C, int lane, const float* __restrict__ gamma,
                                                const float* __restrict__ beta) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < PER; ++i) s += (lane + 32 * i < C) ? v[i] : 0.f;
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    float d = (lane + 32 * i < C) ? v[i] - mean : 0.f;
    q += d * d;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)C + 1e-5f);
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    int c = lane + 32 * i;
    if (c < C) v[i] = (v[i] - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c);
  }
}

__global__ void __launch_bounds__(256) layer_norm_kernel(const float* __restrict__ x, int64_t ldx,
                                                         float* __restrict__ y, int64_t ldy,
                                                         const float* __restrict__ gamma,
                                                         const float* __restrict__ beta, int64_t M, int C) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int64_t m = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (m >= M) return;
  float v[LN_MAX_PER_LANE];
  const float* xr = x + m * ldx;
#pragma unroll
  for (int i = 0; i < LN_MAX_PER_LANE; ++i) {
    int c = lane + 32 * i;
    v[i] = c < C ? xr[c] : 0.f;
  }
  warp_layer_norm<LN_MAX_PER_LANE>(v, C, lane, gamma, beta);
  float* yr = y + m * ldy;
#pragma unroll
  for (int i = 0; i < LN_MAX_PER_LANE; ++i) {
    int c = lane + 32 * i;
    if (c < C) yr[c] = v[i];
  }
}

// One warp = `run_len` consecutive tokens of one utterance (chosen by the launcher so that the grid is whole waves).  The lane keeps its channels of the last
// k-1 normalised rows in registers (a sliding window), so every input row is read once, every
// output row written once, and nothing goes through shared memory.  The k-1 rows before the run
// are re-normalised by the warp (halo).  Rows are fetched two iterations ahead of their use so the
// global-load latency overlaps the arithmetic of the rows in between.
constexpr int MAXK = 8;
constexpr int DW_PER = 6;   // channels per lane: C <= 192

template <int K>
__global__ void __launch_bounds__(128) ln_dwconv_kernel(const float* __restrict__ x, float* __restrict__ u,
                                                        const float* __restrict__ gamma,
                                                        const float* __restrict__ beta,
                                                        const float* __restrict__ w,
                                                        const float* __restrict__ bias, int64_t L, int C,
                                                        int run_len) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int64_t run = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
  const int64_t b = blockIdx.y;
  const int64_t t0 = run * run_len;
  if (t0 >= L) return;
  float wv[DW_PER][K], bv[DW_PER], gv[DW_PER], be[DW_PER];
#pragma unroll
  for (int i = 0; i < DW_PER; ++i) {
    const int c = lane + 32 * i;
    const bool ok = c < C;
    bv[i] = ok ? __ldg(bias + c) : 0.f;
    gv[i] = ok ? __ldg(gamma + c) : 0.f;
    be[i] = ok ? __ldg(beta + c) : 0.f;
#pragma unroll
    for (int j = 0; j < K; ++j) wv[i][j] = ok ? __ldg(w + c * K + j) : 0.f;
  }
  float win[K][DW_PER];   // win[j] = normalised row t - (K-1) + j ; zero before the utterance starts
#pragma unroll
  for (int j = 0; j < K; ++j)
#pragma unroll
    for (int i = 0; i < DW_PER; ++i) win[j][i] = 0.f;

  const float invC = 1.0f / (float)C;
  const int64_t tend = (t0 + run_len < L) ? t0 + run_len : L;
  const float* xb = x + b * L * C;
  auto fetch = [&](int64_t t, float (&dst)[DW_PER]) {
#pragma unroll
    for (int i = 0; i < DW_PER; ++i) {
      const int c = lane + 32 * i;
      dst[i] = (t >= 0 && t < tend && c < C) ? __ldg(xb + t * C + c) : 0.f;
    }
  };
  float r0[DW_PER], r1[DW_PER];     // rows t and t+1, in flight
  fetch(t0 - (K - 1), r0);
  fetch(t0 - (K - 1) + 1, r1);
  for (int64_t t = t0 - (K - 1); t < tend; ++t) {
    if (t == tend - 1) pdl_trigger();     // a single-wave grid at long utterances: let the next kernel in only at the end
    float v[DW_PER];
#pragma unroll
    for (int i = 0; i < DW_PER; ++i) { v[i] = r0[i]; r0[i] = r1[i]; }
    fetch(t + 2, r1);
    // slide
#pragma unroll
    for (int j = 0; j + 1 < K; ++j)
#pragma unroll
      for (int i = 0; i < DW_PER; ++i) win[j][i] = win[j + 1][i];
    if (t >= 0) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < DW_PER; ++i) s += v[i];
      const float mean = warp_sum(s) * invC;
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < DW_PER; ++i) {
        const float d = (lane + 32 * i < C) ? v[i] - mean : 0.f;
        q += d * d;
      }
      const float rstd = rsqrtf(warp_sum(q) * invC + 1e-5f);
#pragma unroll
      for (int i = 0; i < DW_PER; ++i) win[K - 1][i] = (v[i] - mean) * rstd * gv[i] + be[i];
    } else {
#pragma unroll
      for (int i = 0; i < DW_PER; ++i) win[K - 1][i] = 0.f;
    }
    if (t >= t0) {
      float* ur = u + (b * L + t) * C;
#pragma unroll
      for (int i = 0; i < DW_PER; ++i) {
        const int c = lane + 32 * i;
        float acc = bv[i];
#pragma unroll
        for (int j = 0; j < K; ++j) acc = fmaf(wv[i][j], win[j][i], acc);
        if (c < C) ur[c] = acc;
      }
    }
  }
}

}  // namespace

cudaError_t launch_layer_norm(const float* x, int64_t ldx, float* y, int64_t ldy, const float* gamma,
                              const float* beta, int64_t M, int C, cudaStream_t s, int64_t* launches) {
  if (M <= 0) return cudaSuccess;
  if (C > 32 * LN_MAX_PER_LANE) return cudaErrorInvalidValue;
  const cudaError_t e = launch_k(layer_norm_kernel, dim3((unsigned)((M + 7) / 8)), dim3(256), 0, s, x, ldx, y, ldy, gamma,
                                 beta, M, C);
  if (launches) ++*launches;
  return e;
}

cudaError_t launch_ln_dwconv(const float* x, float* u, const float* gamma, const float* beta, const float* w,
                             const float* bias, int64_t B, int64_t L, int C, int k, cudaStream_t s,
                             int64_t* launches, int run_len, int* run_len_used) {
  if (B <= 0 || L <= 0) return cudaSuccess;
  if (C > 32 * DW_PER || k < 1 || k > MAXK || B > 65535 || run_len < 0) return cudaErrorInvalidValue;
  // Run length: a warp re-normalises the k - 1 rows before its run, so its cost is run + k - 1 rows, and the grid
  // runs in waves of (resident CTAs per SM) x SMs.  At config 2 runs of 16 tokens gave 768 CTAs for 592 resident
  // ones — a second wave of 176 — where runs of 21 give one wave of 576 (24 rows per warp instead of 2 x 19).
  // A given run_len > 0 replaces the rule (the result does not depend on it: tests place run boundaries with it).
  if (run_len == 0) {
    static int slots = 0;
    if (slots == 0) {
      int dev = 0, sms = 148, occ = 4;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ln_dwconv_kernel<4>, 128, 0) != cudaSuccess || occ < 1) occ = 4;
      slots = occ * sms;
    }
    run_len = 16;
    int64_t best = -1;
    for (int r = 4; r <= 64; ++r) {
      const int64_t ctas = B * (((L + r - 1) / r + 3) / 4);
      const int64_t cost = ((ctas + slots - 1) / slots) * (r + k - 1);
      if (best < 0 || cost < best) { best = cost; run_len = r; }
    }
  }
  if (run_len_used) *run_len_used = run_len;
  const int64_t runs = (L + run_len - 1) / run_len;
  dim3 grid((unsigned)((runs + 3) / 4), (unsigned)B);
  cudaError_t e_launch = cudaSuccess;
  switch (k) {
#define VASR_DW_CASE(KK) case KK: e_launch = launch_k(ln_dwconv_kernel<KK>, grid, dim3(128), 0, s, x, u, gamma, beta, w, bias, L, C, run_len); break;
    VASR_DW_CASE(1) VASR_DW_CASE(2) VASR_DW_CASE(3) VASR_DW_CASE(4)
    VASR_DW_CASE(5) VASR_DW_CASE(6) VASR_DW_CASE(7) VASR_DW_CASE(8)
#undef VASR_DW_CASE
  }
  if (launches) ++*launches;
  return e_launch;
}

}  // namespace vasr
