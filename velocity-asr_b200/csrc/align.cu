// align.cu — CTC forced alignment (Viterbi) and transcript log-likelihood on the device (include/vasr.h states
// the rule).  One CTA per utterance walks its frames in order; thread i owns the states [i E, (i+1) E) of the
// expansion blank, y0, blank, y1, ..., blank and keeps their scores (fp64) in one array, in shared memory when it
// fits, else in global scratch (the same code through a generic pointer, so a long target has no cap but memory).
//
// The array is updated in place: inside its own range a thread walks the states downwards, so delta[s-1] and
// delta[s-2] still hold the previous frame when state s reads them.  The two states below a range belong to the
// thread before it (E >= 2); each thread publishes its two top states in a boundary slot at the end of a frame, and
// the slots alternate between frames, so one barrier per frame orders everything.
//
// Viterbi: per state and frame a 2-bit backpointer (0 stay, 1 from s-1, 2 from s-2), 16 to a 32-bit word; E is a
// multiple of 16, so every word has one writer.  Thread 0 then walks the pointers back from the final state.
#include <float.h>

#include "common.cuh"
#include "kernels.cuh"

namespace vasr {

namespace {

struct AlignArgs {
  const float* logits;       // (B, L, V)
  const float2* stats;       // (B * L) (max, log sum exp(x - max)) from launch_beam_rows; NULL: logits are log-probs
  int64_t L;
  int V, blank;
  const int32_t* lens;       // frames of utterance b at lens[b * lens_stride]; NULL: L
  int lens_stride;
  const int32_t* targets;    // (B, U_max)
  const int32_t* target_lens;
  int64_t U_max;
  int E;                     // states per thread
  double* delta_g;           // (B, E * blockDim) global scores, or NULL: in shared memory after the boundary slots
  uint32_t* bp;              // Viterbi: (B, L, words) backpointers
  int64_t words;
  int32_t* out_labels;       // Viterbi: (B, L)
  float* out_lp;             // Viterbi: (B, L)
  double* out_score;         // (B)
};

template <bool kViterbi>
__global__ void __launch_bounds__(512, 1) ctc_align_kernel(const AlignArgs a) {
  extern __shared__ double smem[];
  const int64_t b = blockIdx.x;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int64_t Lb = a.lens ? (int64_t)a.lens[b * a.lens_stride] : a.L;
  const int64_t U = a.target_lens[b];
  const int64_t S = 2 * U + 1;
  const int32_t* y = a.targets + b * a.U_max;
  double2* bnd = reinterpret_cast<double2*>(smem);   // [2][nt]: (delta[top], delta[top - 1]) of each thread's range
  double* delta = a.delta_g ? a.delta_g + b * (int64_t)a.E * nt : smem + 4 * nt;
  const int64_t s0 = (int64_t)tid * a.E, s1 = s0 + a.E < S ? s0 + a.E : S;
  const double NEG = -INFINITY;

  // frame -1: only state 0 (score 0), so frame 0 starts in blank or in y0
  for (int64_t s = s0; s < s1; ++s) delta[s] = s == 0 ? 0.0 : NEG;
  bnd[tid] = make_double2(s0 + a.E - 1 == 0 ? 0.0 : NEG, s0 + a.E - 2 == 0 ? 0.0 : NEG);
  __syncthreads();

  auto label = [&](int64_t s) -> int { return (s & 1) ? __ldg(y + (s >> 1)) : a.blank; };
  for (int64_t t = 0; t < Lb; ++t) {
    const int p = (int)(t & 1);
    const int64_t row = b * a.L + t;
    const float* x = a.logits + row * a.V;
    const float2 st = a.stats ? a.stats[row] : make_float2(0.f, 0.f);
    const double2 left = tid > 0 ? bnd[p * nt + tid - 1] : make_double2(NEG, NEG);   // delta[s0 - 1], delta[s0 - 2]
    auto old = [&](int64_t i) -> double { return i >= s0 ? delta[i] : i == s0 - 1 ? left.x : left.y; };
    double top1 = NEG, top2 = NEG;
    if (s0 < S) {
      double c0 = delta[s1 - 1], c1 = old(s1 - 2), c2 = old(s1 - 3);
      uint32_t word = 0;
      int ynext = -1;   // walking down, the id below an odd state is the label of the next odd state: one load each
      for (int64_t s = s1 - 1; s >= s0; --s) {
        int lab = a.blank;
        bool skip = false;
        if (s & 1) {
          lab = ynext >= 0 ? ynext : __ldg(y + (s >> 1));
          ynext = s >= 3 ? __ldg(y + (s >> 1) - 1) : -1;
          skip = s >= 3 && lab != ynext;
        }
        const float xf = __ldg(x + lab);
        const double lp = (double)(a.stats ? (xf - st.x) - st.y : xf);
        double v;
        if (kViterbi) {
          double best = c0;
          uint32_t arg = 0;
          if (c1 > best) best = c1, arg = 1;
          if (skip && c2 > best) best = c2, arg = 2;
          v = best + lp;
          word |= arg << (2 * (s & 15));
          if ((s & 15) == 0) {
            a.bp[row * a.words + (s >> 4)] = word;
            word = 0;
          }
        } else {
          double m = c0;
          if (c1 > m) m = c1;
          if (skip && c2 > m) m = c2;
          if (m == NEG) {
            v = NEG;
          } else {
            double sum = exp(c0 - m) + exp(c1 - m);
            if (skip) sum += exp(c2 - m);
            v = (m + log(sum)) + lp;
          }
        }
        delta[s] = v;
        if (s == s0 + a.E - 1) top1 = v;
        if (s == s0 + a.E - 2) top2 = v;
        c0 = c1;
        c1 = c2;
        c2 = s - 3 >= 0 ? old(s - 3) : NEG;
      }
    }
    bnd[(p ^ 1) * nt + tid] = make_double2(top1, top2);
    __syncthreads();
  }

  // the end: state 2U (trailing blank) or 2U - 1 (last token); every thread reads the result
  const double last = U > 0 ? delta[2 * U - 1] : NEG, tail = delta[2 * U];
  double score;
  int64_t fin = 2 * U;
  if (kViterbi) {
    if (U > 0 && !(tail > last)) fin = 2 * U - 1;
    score = fin == 2 * U ? tail : last;
  } else {
    const double m = last > tail ? last : tail;
    score = m == NEG ? NEG : m + log(exp(last - m) + exp(tail - m));
  }
  if (tid == 0) a.out_score[b] = score;
  if (!kViterbi) return;

  int32_t* lab_out = a.out_labels + b * a.L;
  float* lp_out = a.out_lp + b * a.L;
  const bool found = score != NEG;
  for (int64_t t = found ? Lb + tid : tid; t < a.L; t += nt) {   // padding frames, and every frame without a path
    lab_out[t] = -1;
    lp_out[t] = 0.f;
  }
  if (!found || tid != 0) return;
  int64_t s = fin;
  for (int64_t t = Lb - 1; t >= 0; --t) {
    const int64_t row = b * a.L + t;
    const int lab = label(s);
    const float xf = a.logits[row * a.V + lab];
    float lp = xf;
    if (a.stats) {
      const float2 st = a.stats[row];
      lp = (xf - st.x) - st.y;
    }
    lab_out[t] = lab;
    lp_out[t] = lp;
    s -= (a.bp[row * a.words + (s >> 4)] >> (2 * (s & 15))) & 3u;
  }
}

}  // namespace

int64_t ctc_align_words(int64_t U) { return (2 * U + 1 + 15) / 16; }

void ctc_align_layout(int64_t U, bool viterbi, int* threads, int* E) {
  const int64_t g = viterbi ? 16 : 2, units = (2 * U + 1 + g - 1) / g;
  const int64_t nt = ((units + 31) / 32) * 32;
  *threads = (int)(nt < 512 ? nt : 512);
  *E = (int)(g * ((units + *threads - 1) / *threads));
}

size_t ctc_align_smem(int threads, int E, bool delta_in_smem) {
  return (size_t)threads * 4 * sizeof(double) + (delta_in_smem ? (size_t)threads * E * sizeof(double) : 0);
}

cudaError_t launch_ctc_align(const float* logits, const float2* stats, int64_t B, int64_t L, int V, int blank,
                             const int32_t* lens, int lens_stride, const int32_t* targets, int64_t U_max,
                             const int32_t* target_lens, int threads, int E, double* delta_g, uint32_t* bp,
                             int64_t words, int32_t* out_labels, float* out_lp, double* out_score, cudaStream_t s) {
  if (B <= 0) return cudaSuccess;
  AlignArgs a{logits, stats, L, V, blank, lens, lens_stride, targets, target_lens, U_max, E, delta_g, bp, words,
              out_labels, out_lp, out_score};
  const size_t smem = ctc_align_smem(threads, E, delta_g == nullptr);
  if (bp) {
    cudaError_t e = cudaFuncSetAttribute(ctc_align_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    ctc_align_kernel<true><<<(unsigned)B, threads, smem, s>>>(a);
  } else {
    cudaError_t e = cudaFuncSetAttribute(ctc_align_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    ctc_align_kernel<false><<<(unsigned)B, threads, smem, s>>>(a);
  }
  return cudaGetLastError();
}

}  // namespace vasr
