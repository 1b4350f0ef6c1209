// mel.cu — log-mel front end (compute_mel_spectrogram, velocity_asr/audio.py:65-143).
//
// Stage order of the reference: reflect-pad 200 (audio.py:100-101) -> frames of 400 every 160
// with a periodic Hann window -> one-sided 400-point DFT (torch.stft, audio.py:104-112) ->
// power (:115) -> 80 x 201 HTK-mel filterbank (:118-126) -> log(. + 1e-10) (:129) ->
// per (utterance, bin) (x - mean_T) / (std_T unbiased + 1e-10) (:132-135) -> (B, T, 80).
//
// Structure: ONE pass from PCM to log-mel (mel_fft_kernel).  A CTA stages the samples of 32
// consecutive frames of one utterance in shared memory (reflect padding is index arithmetic, the
// padded signal is never materialised); each warp then takes a frame at a time through a
// 400-point FFT, the power spectrum, the band-sparse mel filterbank and the log, and the CTA
// leaves (mean, M2) partials of its frames for the per-utterance normalisation.  A true 400-point
// transform, not a zero-padded 512-point one: the bin spacing has to be 40 Hz to match the
// reference (SURVEY.md section 0.3).
//
// The FFT.  400 = 20 x 20 (Cooley-Tukey): lane q < 20 transforms the 20 samples x[20 n1 + q]
// (windowed on load), multiplies by the twiddles W400^(q k1) and leaves column q of a 20 x 20
// matrix in shared memory; lane k1 then transforms row k1 and holds X[k1 + 20 k2].  Each 20-point
// transform runs in registers as a Good-Thomas 4 x 5 prime-factor transform (no inner twiddles).
// ~13 kflop per frame instead of the 322 kflop of the dense DFT the first version ran as a GEMM
// (1.42 ms of an 11 ms step at config 2); fp32 throughout, error ~1e-6, well inside the 1e-4 bar.
#include "common.cuh"
#include "kernels.cuh"

namespace vasr {

namespace {

// ---- 20-point DFT in registers: Good-Thomas with N = 4 x 5 ---------------------------------
// in[n], n = (5 n1 + 4 n2) mod 20  ->  out[k], k = (5 k1 + 16 k2) mod 20  (CRT: k = k1 mod 4, k2 mod 5)
__device__ __forceinline__ void dft5(float (&r)[5], float (&i)[5]) {
  constexpr float C1 = 0.30901699437494742f, C2 = -0.80901699437494742f;
  constexpr float S1 = 0.95105651629515357f, S2 = 0.58778525229247313f;
  const float t1r = r[1] + r[4], t1i = i[1] + i[4], t2r = r[2] + r[3], t2i = i[2] + i[3];
  const float t3r = r[1] - r[4], t3i = i[1] - i[4], t4r = r[2] - r[3], t4i = i[2] - i[3];
  const float a1r = r[0] + C1 * t1r + C2 * t2r, a1i = i[0] + C1 * t1i + C2 * t2i;
  const float a2r = r[0] + C2 * t1r + C1 * t2r, a2i = i[0] + C2 * t1i + C1 * t2i;
  const float b1r = S1 * t3r + S2 * t4r, b1i = S1 * t3i + S2 * t4i;
  const float b2r = S2 * t3r - S1 * t4r, b2i = S2 * t3i - S1 * t4i;
  r[0] = r[0] + t1r + t2r;  i[0] = i[0] + t1i + t2i;
  r[1] = a1r + b1i;  i[1] = a1i - b1r;      // a1 - i b1
  r[4] = a1r - b1i;  i[4] = a1i + b1r;      // a1 + i b1
  r[2] = a2r + b2i;  i[2] = a2i - b2r;
  r[3] = a2r - b2i;  i[3] = a2i + b2r;
}
__device__ __forceinline__ void dft4(float (&r)[4], float (&i)[4]) {
  const float s02r = r[0] + r[2], s02i = i[0] + i[2], d02r = r[0] - r[2], d02i = i[0] - i[2];
  const float s13r = r[1] + r[3], s13i = i[1] + i[3], d13r = r[1] - r[3], d13i = i[1] - i[3];
  r[0] = s02r + s13r;  i[0] = s02i + s13i;
  r[2] = s02r - s13r;  i[2] = s02i - s13i;
  r[1] = d02r + d13i;  i[1] = d02i - d13r;  // d02 - i d13
  r[3] = d02r - d13i;  i[3] = d02i + d13r;  // d02 + i d13
}
__device__ __forceinline__ void dft20(float (&re)[20], float (&im)[20]) {
  float cr[4][5], ci[4][5];
#pragma unroll
  for (int n1 = 0; n1 < 4; ++n1) {
    float r[5], i[5];
#pragma unroll
    for (int n2 = 0; n2 < 5; ++n2) { r[n2] = re[(5 * n1 + 4 * n2) % 20]; i[n2] = im[(5 * n1 + 4 * n2) % 20]; }
    dft5(r, i);
#pragma unroll
    for (int k2 = 0; k2 < 5; ++k2) { cr[n1][k2] = r[k2]; ci[n1][k2] = i[k2]; }
  }
#pragma unroll
  for (int k2 = 0; k2 < 5; ++k2) {
    float r[4], i[4];
#pragma unroll
    for (int n1 = 0; n1 < 4; ++n1) { r[n1] = cr[n1][k2]; i[n1] = ci[n1][k2]; }
    dft4(r, i);
#pragma unroll
    for (int k1 = 0; k1 < 4; ++k1) { re[(5 * k1 + 16 * k2) % 20] = r[k1]; im[(5 * k1 + 16 * k2) % 20] = i[k1]; }
  }
}

constexpr int MEL_WARPS = 8, FPW = 4, FPC = MEL_WARPS * FPW;   // 32 frames per CTA
constexpr int NFFT = 400, NHOP = 160, NPAD = 200, NBIN = 201;
constexpr int TLD = 21;                                        // row stride of the 20 x 20 exchange matrix
constexpr int MAX_MELS = 128;
constexpr int NX = NHOP * (FPC - 1) + NFFT;
inline size_t mel_fft_smem(int n_mels) {
  return sizeof(float) * (size_t)(2 * NFFT + NFFT + NX + MEL_WARPS * 2 * 20 * TLD + FPC * n_mels);
}

// tw: W400^m = (cos, -sin)(2 pi m / 400), m in [0, 400); win: the 400-tap analysis window.
// raw (B, T, n_mels) <- log(mel power + 1e-10); part (B, nblk, n_mels, 2) <- (mean, M2) of the
// CTA's frames (NULL to skip).
__global__ void __launch_bounds__(MEL_WARPS * 32) mel_fft_kernel(
    const float* __restrict__ pcm, float* __restrict__ raw, double* __restrict__ part, int64_t S, int64_t T,
    int n_mels, const int* __restrict__ fb_lo, const int* __restrict__ fb_off, const float* __restrict__ fb_w,
    const float* __restrict__ win, const float2* __restrict__ tw, const int32_t* __restrict__ rag) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) float mel_smem[];
  float2* s_tw = reinterpret_cast<float2*>(mel_smem);                  // NFFT float2
  float* s_win = mel_smem + 2 * NFFT;                                  // NFFT
  float* s_x = s_win + NFFT;                                           // NX samples of FPC frames
  float* s_t = s_x + NX;                                               // per warp: re | im of the 20 x 20 matrix
  float* s_lm = s_t + MEL_WARPS * 2 * 20 * TLD;                        // FPC x n_mels log-mel values

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t b = blockIdx.y;
  const int64_t t0 = (int64_t)blockIdx.x * FPC;
  // ragged batch: this utterance has Sb <= S samples / Tb <= T frames; rows keep the strides of S and T
  const int64_t Sb = rag ? rag[b * RAG_STRIDE + RAG_S] : S;
  const int64_t Tb = rag ? rag[b * RAG_STRIDE + RAG_T] : T;
  if (Tb <= t0) return;                                        // whole CTA past the utterance's end
  const int nfr = (int)((Tb - t0) < FPC ? (Tb - t0) : FPC);   // frames of this CTA that exist
  const float* xb = pcm + b * S;
  const int nsamp = NHOP * (nfr - 1) + NFFT;
  // The samples of the CTA's frames: contiguous in the signal except where the reflect padding folds them back at
  // either end of the utterance (audio.py:100-101).  Interior CTAs — all but the first and the last one or two of an
  // utterance — copy them as 16-byte vectors (the window start (t0 * 160 - 200) * 4 B is a multiple of 16 whenever
  // the utterance's row is: S % 4 == 0).
  const int64_t g0 = t0 * NHOP - NPAD;
  if (g0 >= 0 && g0 + nsamp <= Sb && ((reinterpret_cast<uintptr_t>(xb + g0) & 15) == 0) && (nsamp & 3) == 0) {
    const float4* src = reinterpret_cast<const float4*>(xb + g0);
    float4* dst = reinterpret_cast<float4*>(s_x);
    for (int i = tid; i < nsamp / 4; i += MEL_WARPS * 32) dst[i] = __ldg(src + i);
  } else {
    for (int i = tid; i < nsamp; i += MEL_WARPS * 32) {
      int64_t g = g0 + i;                         // index into the unpadded signal
      if (g < 0) g = -g;                          // reflect without repeating the edge sample
      if (g >= Sb) g = 2 * (Sb - 1) - g;
      s_x[i] = (g >= 0 && g < Sb) ? __ldg(xb + g) : 0.f;
    }
  }
  for (int i = tid; i < NFFT; i += MEL_WARPS * 32) {
    s_win[i] = __ldg(win + i);
    s_tw[i] = __ldg(tw + i);
  }
  __syncthreads();

  float* tr = s_t + warp * 2 * 20 * TLD;
  float* ti = tr + 20 * TLD;
  float* pw = tr;                                // the power spectrum reuses the matrix once it is in registers
  for (int fi = 0; fi < FPW; ++fi) {
    const int f = warp * FPW + fi;
    if (f >= nfr) break;                         // warp-uniform
    const float* xf = s_x + NHOP * f;
    if (lane < 20) {
      const int q = lane;
      float re[20], im[20];
#pragma unroll
      for (int n1 = 0; n1 < 20; ++n1) {
        re[n1] = xf[20 * n1 + q] * s_win[20 * n1 + q];
        im[n1] = 0.f;
      }
      dft20(re, im);
#pragma unroll
      for (int k1 = 0; k1 < 20; ++k1) {
        const float2 w = s_tw[(q * k1) % NFFT];
        tr[k1 * TLD + q] = re[k1] * w.x - im[k1] * w.y;
        ti[k1 * TLD + q] = re[k1] * w.y + im[k1] * w.x;
      }
    }
    __syncwarp();
    if (lane < 20) {
      const int k1 = lane;
      float re[20], im[20];
#pragma unroll
      for (int n2 = 0; n2 < 20; ++n2) { re[n2] = tr[k1 * TLD + n2]; im[n2] = ti[k1 * TLD + n2]; }
      dft20(re, im);
      __syncwarp(0x000fffffu);                   // every row is in registers before pw overwrites the matrix
#pragma unroll
      for (int k2 = 0; k2 <= 10; ++k2) {
        const int k = k1 + 20 * k2;
        if (k < NBIN) pw[k] = re[k2] * re[k2] + im[k2] * im[k2];
      }
    }
    __syncwarp();
    for (int j = lane; j < n_mels; j += 32) {
      const int lo = fb_lo[j], o0 = fb_off[j], o1 = fb_off[j + 1];
      float acc = 0.f;
      for (int o = o0; o < o1; ++o) acc = fmaf(__ldg(fb_w + o), pw[lo + (o - o0)], acc);
      const float v = logf(acc + 1e-10f);
      raw[((b * T + t0 + f) * n_mels) + j] = v;
      s_lm[f * n_mels + j] = v;
    }
    __syncwarp();
  }
  if (part == nullptr) return;
  __syncthreads();
  // (mean, M2) of this CTA's frames per mel bin; mel_stats_combine merges the partials in frame order
  for (int j = tid; j < n_mels; j += MEL_WARPS * 32) {
    double sum = 0.0;
    for (int f = 0; f < nfr; ++f) sum += (double)s_lm[f * n_mels + j];
    const double mu = sum / (double)nfr;
    double m2 = 0.0;
    for (int f = 0; f < nfr; ++f) {
      const double d = (double)s_lm[f * n_mels + j] - mu;
      m2 += d * d;
    }
    double* o = part + ((b * gridDim.x + blockIdx.x) * n_mels + j) * 2;
    o[0] = mu;
    o[1] = m2;
  }
}

// Normalisation into the layout the temporal-binding projection reads.  With `part` the CTA first merges the
// per-CTA (mean, M2) partials of mel_fft_kernel for its utterance into mean and 1 / (unbiased std + 1e-10)
// (audio.py:132-135), fp64, in a fixed order — every CTA of an utterance computes the same bits.  Two
// division-free passes (grand mean, then sum of M2_k + n_k (mean_k - mean)^2): the first version
// was a separate one-CTA-per-utterance kernel running Chan's update block by block, two fp64 divisions inside a
// dependent chain of 47 steps — 28 us on the critical path for 5,120 numbers.
__global__ void __launch_bounds__(256) mel_finish_kernel(const float* __restrict__ raw,
                                                         const double* __restrict__ part, int nblk,
                                                         float* __restrict__ out, int64_t T, int n_mels, int64_t fpu,
                                                         int front, const int32_t* __restrict__ rag, int per_cta) {
  __shared__ float s_mean[MAX_MELS], s_rstd[MAX_MELS];
  pdl_trigger();
  pdl_wait();
  const int64_t b = blockIdx.y;
  const int64_t Tb = rag ? rag[b * RAG_STRIDE + RAG_T] : T;   // the partials keep the row stride nblk of the longest
  const bool norm = part != nullptr;
  if (norm) {
    // threads (j, g): mel bin j, every G-th block starting at g — the loads of a pass are in flight together, the
    // G partial sums of a bin are added in the order of g (the same bits in every CTA of the utterance)
    __shared__ double s_acc[256];
    const int G = 256 / n_mels < 1 ? 1 : (256 / n_mels > 4 ? 4 : 256 / n_mels);
    const int j = threadIdx.x % n_mels, g = threadIdx.x / n_mels;
    const bool on = g < G;
    const int nb = (int)((Tb + FPC - 1) / FPC);
    const double last_n = (double)(Tb - (int64_t)(nb - 1) * FPC);
    const double* p = part + (b * nblk * n_mels + j) * 2;
    const int64_t st = 2 * n_mels;
    double s = 0.0;
    if (on) {
#pragma unroll 8
      for (int k = g; k < nb; k += G) s += (k == nb - 1 ? last_n : (double)FPC) * p[k * st];
    }
    s_acc[threadIdx.x] = s;
    __syncthreads();
    double tot = 0.0;
    for (int q = 0; q < G; ++q) tot += s_acc[q * n_mels + j];
    const double mu = tot / (double)Tb;
    __syncthreads();
    double m2 = 0.0;
    if (on) {
#pragma unroll 8
      for (int k = g; k < nb; k += G) {
        const double2 pk = *reinterpret_cast<const double2*>(p + k * st);
        const double d = pk.x - mu;
        m2 += pk.y + (k == nb - 1 ? last_n : (double)FPC) * d * d;
      }
    }
    s_acc[threadIdx.x] = m2;
    __syncthreads();
    if (g == 0) {
      double m2t = 0.0;
      for (int q = 0; q < G; ++q) m2t += s_acc[q * n_mels + j];
      // torch.std(unbiased) of a single frame is NaN; keep that behaviour (0/0).
      const double sd = sqrt(m2t / (double)(Tb - 1));
      s_mean[j] = (float)mu;
      s_rstd[j] = (float)(1.0 / (sd + 1e-10));
    }
    __syncthreads();
  }
  const uint32_t total = (uint32_t)(fpu * n_mels);            // checked by the launcher to fit
  const uint32_t i0 = blockIdx.x * (uint32_t)per_cta;
  const uint32_t i1 = i0 + (uint32_t)per_cta < total ? i0 + (uint32_t)per_cta : total;
  const float* rb = raw + b * T * n_mels;
  float* ob = out + b * (int64_t)total;
  if ((n_mels & 3) == 0 && (reinterpret_cast<uintptr_t>(rb) & 15) == 0 && (reinterpret_cast<uintptr_t>(ob) & 15) == 0) {
    // four mel bins of one frame per thread and access (a group never straddles a frame: n_mels % 4 == 0)
#pragma unroll 4
    for (uint32_t idx = i0 + 4 * threadIdx.x; idx < i1; idx += 1024) {
      const uint32_t p = idx / (uint32_t)n_mels;
      const uint32_t j = idx - p * (uint32_t)n_mels;
      const int64_t t = (int64_t)p - front;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t >= 0 && t < Tb) {
        v = __ldg(reinterpret_cast<const float4*>(rb + t * n_mels + j));
        if (norm) {
          v.x = (v.x - s_mean[j]) * s_rstd[j];
          v.y = (v.y - s_mean[j + 1]) * s_rstd[j + 1];
          v.z = (v.z - s_mean[j + 2]) * s_rstd[j + 2];
          v.w = (v.w - s_mean[j + 3]) * s_rstd[j + 3];
        }
      }
      *reinterpret_cast<float4*>(ob + idx) = v;
    }
    return;
  }
  for (uint32_t idx = i0 + threadIdx.x; idx < i1; idx += 256) {
    const uint32_t p = idx / (uint32_t)n_mels;
    const uint32_t j = idx - p * (uint32_t)n_mels;
    const int64_t t = (int64_t)p - front;
    float v = 0.f;
    if (t >= 0 && t < Tb) {
      v = rb[t * n_mels + j];
      if (norm) v = (v - s_mean[j]) * s_rstd[j];
    }
    ob[idx] = v;
  }
}

}  // namespace

int64_t mel_fft_blocks(int64_t T) { return (T + FPC - 1) / FPC; }

cudaError_t launch_mel_fft(const float* pcm, float* raw, double* part, int64_t B, int64_t S, int64_t T, int n_mels,
                           const int* fb_lo, const int* fb_off, const float* fb_w, const float* win,
                           const float* tw, cudaStream_t s, int64_t* launches, const int32_t* rag) {
  if (B <= 0 || T <= 0) return cudaSuccess;
  if (B > 65535 || n_mels > MAX_MELS || S <= NPAD) return cudaErrorInvalidValue;
  dim3 grid((unsigned)mel_fft_blocks(T), (unsigned)B);
  const size_t smem = mel_fft_smem(n_mels);
  cudaError_t e = cudaFuncSetAttribute(mel_fft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  e = launch_k(mel_fft_kernel, grid, dim3(MEL_WARPS * 32), smem, s, pcm, raw, part, S, T, n_mels, fb_lo, fb_off, fb_w, win,
               reinterpret_cast<const float2*>(tw), rag);
  if (launches) ++*launches;
  return e;
}

cudaError_t launch_mel_finish(const float* raw, float* out, int64_t B,
                              int64_t T, int n_mels, int64_t frames_per_utt, int front, cudaStream_t s,
                              int64_t* launches, const int32_t* rag, const double* part) {
  if (B <= 0) return cudaSuccess;
  if (B > 65535 || n_mels > MAX_MELS) return cudaErrorInvalidValue;
  // a CTA takes 8 K elements, or 1/128 of a long utterance (every CTA of an utterance repeats the merge of its partials)
  const int64_t total = frames_per_utt * n_mels;
  if (total >= (1LL << 31)) return cudaErrorInvalidValue;
  int64_t per_cta = total / 128 > 8192 ? total / 128 : 8192;
  per_cta = (per_cta + 1023) / 1024 * 1024;
  dim3 grid((unsigned)((total + per_cta - 1) / per_cta), (unsigned)B);
  const cudaError_t e = launch_k(mel_finish_kernel, grid, dim3(256), 0, s, raw, part, (int)mel_fft_blocks(T), out,
                                 T, n_mels, frames_per_utt, front, rag, (int)per_cta);
  if (launches) ++*launches;
  return e;
}

}  // namespace vasr
