// ctc.cu — CTC greedy decode on the device (ctc_greedy_decode, velocity_asr/decode.py:27-71):
// argmax over the vocabulary (ties -> lowest index, as torch.argmax) and the blank/repeat
// collapse, which the reference does in a host Python loop after a D2H `.tolist()`.
// Integer work; results are bit-exact by construction.
#include "common.cuh"
#include "kernels.cuh"

namespace vasr {

namespace {

// one warp per token row
__global__ void __launch_bounds__(256) argmax_kernel(const float* __restrict__ logits, int32_t* __restrict__ pred,
                                                     int64_t M, int V) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int64_t m = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (m >= M) return;
  const float* r = logits + m * V;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int n = lane; n < V; n += 32) {
    const float v = r[n];
    if (v > best || (bi == 0x7fffffff)) {  // first element seen always wins; later only strictly greater
      best = v;
      bi = n;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > best || (ov == best && oi < bi)) {
      best = ov;
      bi = oi;
    }
  }
  if (lane == 0) pred[m] = bi == 0x7fffffff ? 0 : bi;
}

// one warp per utterance: keep[t] = pred[t] != blank && (!collapse || t == 0 || pred[t] != pred[t-1]).
// (A blank resets the reference's `prev`, and a blank predecessor differs from any kept token,
// so comparing with the raw predecessor is the same rule, decode.py:55-66.)
// PARTS (256 threads): the frames' predictions are first taken from the per-slot (max, first argmax) pairs the
// CTC-head projection left (GemmArgs::amax_val) — the best over the slots in column order, a later slot only on a
// strictly greater value, i.e. ties -> lowest index as torch.argmax (decode.py:46) — and written to `pred`; warp 0
// then collapses as usual.
template <bool PARTS>
__global__ void __launch_bounds__(PARTS ? 256 : 32) ctc_collapse_kernel(int32_t* pred,
                                                          int32_t* __restrict__ tokens, int32_t* __restrict__ lens,
                                                          int64_t L, int blank, int collapse,
                                                          const int32_t* __restrict__ rag,
                                                          const float* __restrict__ pv, const int32_t* __restrict__ pi,
                                                          int slots, int64_t M) {
  pdl_trigger();
  pdl_wait();
  const int64_t b = blockIdx.x;
  const int lane = threadIdx.x;
  int32_t* p = pred + b * L;
  int32_t* out = tokens + b * L;
  const int64_t Lb = rag ? rag[b * RAG_STRIDE + RAG_L] : L;   // ragged: tokens past the utterance's end are padding
  if (PARTS) {
    for (int64_t t = threadIdx.x; t < Lb; t += 256) {
      float best = -INFINITY;
      int bi = -1;
#pragma unroll 8
      for (int s = 0; s < slots; ++s) {                // unrolled: the slots' loads are independent, the compares are not
        const int i = pi[(int64_t)s * M + b * L + t];
        const float v = pv[(int64_t)s * M + b * L + t];
        if (i >= 0 && (v > best || bi < 0)) { best = v; bi = i; }
      }
      p[t] = bi < 0 ? 0 : bi;
    }
    __syncthreads();
    if (threadIdx.x >= 32) return;
  }
  int count = 0;
  for (int64_t t0 = 0; t0 < Lb; t0 += 32) {
    const int64_t t = t0 + lane;
    int tok = blank;
    bool keep = false;
    if (t < Lb) {
      tok = p[t];
      keep = tok != blank && (!collapse || t == 0 || tok != p[t - 1]);
    }
    const unsigned mask = __ballot_sync(0xffffffffu, keep);
    if (keep) out[count + __popc(mask & ((1u << lane) - 1u))] = tok;
    count += __popc(mask);
  }
  for (int64_t t = count + lane; t < L; t += 32) out[t] = -1;
  if (lane == 0) lens[b] = count;
}

// ctc_greedy_decode_with_timestamps (decode.py:74-125): a token is emitted where a run of equal non-blank
// predictions starts, its (start, end) are the first frame of the run and the first frame after it.  Run
// starts and run ends come in the same order, so both are compacted with the same ballot / popc ranks.
__global__ void __launch_bounds__(32) ctc_runs_kernel(const int32_t* __restrict__ pred, int32_t* __restrict__ tokens,
                                                      int32_t* __restrict__ starts, int32_t* __restrict__ ends,
                                                      int32_t* __restrict__ lens, int64_t L, int blank) {
  const int64_t b = blockIdx.x;
  const int lane = threadIdx.x;
  const int32_t* p = pred + b * L;
  int ns = 0, ne = 0;
  for (int64_t t0 = 0; t0 < L; t0 += 32) {
    const int64_t t = t0 + lane;
    int tok = blank;
    bool st = false, en = false;
    if (t < L) {
      tok = p[t];
      st = tok != blank && (t == 0 || tok != p[t - 1]);
      en = tok != blank && (t == L - 1 || tok != p[t + 1]);
    }
    const unsigned ms = __ballot_sync(0xffffffffu, st), me = __ballot_sync(0xffffffffu, en);
    const unsigned below = (1u << lane) - 1u;
    if (st) {
      const int k = ns + __popc(ms & below);
      tokens[b * L + k] = tok;
      starts[b * L + k] = (int32_t)t;
    }
    if (en) ends[b * L + ne + __popc(me & below)] = (int32_t)(t + 1);
    ns += __popc(ms);
    ne += __popc(me);
  }
  for (int64_t t = ns + lane; t < L; t += 32) {
    tokens[b * L + t] = -1;
    starts[b * L + t] = -1;
    ends[b * L + t] = -1;
  }
  if (lane == 0) lens[b] = ns;
}

// The greedy path with its scores (vasr_ctc_greedy_confidence; include/vasr.h states the rule).  One CTA per
// utterance, over its own frames t < len_b only:
//  1. every thread takes frames: the prediction a_t into pred and lp_t = log softmax(x_t)[a_t] (fp32) into lp;
//     PARTS: from the CTC head's slot partials (GemmArgs::amax_val / amax_idx / amax_sum) — a_t as
//       ctc_collapse_kernel<true> merges them (slot order, a later slot only on a strictly greater value), and
//       Z_t = sum_p sum_p * exp(v_p - max) over the non-empty slots in slot order, lp_t = -log Z_t;
//     else: a_t = pred[t] (argmax_kernel), lp_t = (x_t[a_t] - max) - log sum from beam_rows_kernel's statistics, the
//       fp32 table of the beam search and the forced alignment;
//  2. warp 0 compacts the runs (ctc_runs_kernel's rule, the utterance ending at len_b) while one thread of warp 1
//     adds lp over all frames in time order, in fp64: the greedy path's log-prob;
//  3. each token's thread adds lp over its run [start, end), in time order, in fp64.
template <bool PARTS>
__global__ void __launch_bounds__(256) ctc_confidence_kernel(
    int32_t* pred, float* lp, const float* __restrict__ logits, const float2* __restrict__ stats, int V,
    const float* __restrict__ pv, const int32_t* __restrict__ pi, const float* __restrict__ ps, int slots, int64_t M,
    int32_t* tokens, int32_t* starts, int32_t* ends, double* __restrict__ tok_lp, int32_t* __restrict__ lens,
    double* __restrict__ log_prob, int64_t L, int blank, const int32_t* __restrict__ lens_in, int lens_stride) {
  pdl_trigger();
  pdl_wait();
  __shared__ int s_count;
  const int64_t b = blockIdx.x;
  const int64_t Lb = lens_in ? lens_in[b * lens_stride] : L;
  int32_t* p = pred + b * L;
  float* q = lp + b * L;
  for (int64_t t = threadIdx.x; t < Lb; t += 256) {
    const int64_t row = b * L + t;
    if (PARTS) {
      float best = -INFINITY;
      int bi = -1;
#pragma unroll 8
      for (int s = 0; s < slots; ++s) {
        const int i = pi[(int64_t)s * M + row];
        const float v = pv[(int64_t)s * M + row];
        if (i >= 0 && (v > best || bi < 0)) { best = v; bi = i; }
      }
      float z = 0.f;
#pragma unroll 8
      for (int s = 0; s < slots; ++s)
        if (pi[(int64_t)s * M + row] >= 0) z += ps[(int64_t)s * M + row] * expf(pv[(int64_t)s * M + row] - best);
      p[t] = bi < 0 ? 0 : bi;
      q[t] = -logf(z);
    } else {
      const float2 st = stats[row];
      q[t] = (logits[row * V + p[t]] - st.x) - st.y;
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp == 0) {
    int ns = 0, ne = 0;
    for (int64_t t0 = 0; t0 < Lb; t0 += 32) {
      const int64_t t = t0 + lane;
      int tok = blank;
      bool st = false, en = false;
      if (t < Lb) {
        tok = p[t];
        st = tok != blank && (t == 0 || tok != p[t - 1]);
        en = tok != blank && (t == Lb - 1 || tok != p[t + 1]);
      }
      const unsigned ms = __ballot_sync(0xffffffffu, st), me = __ballot_sync(0xffffffffu, en);
      const unsigned below = (1u << lane) - 1u;
      if (st) {
        const int k = ns + __popc(ms & below);
        tokens[b * L + k] = tok;
        starts[b * L + k] = (int32_t)t;
      }
      if (en) ends[b * L + ne + __popc(me & below)] = (int32_t)(t + 1);
      ns += __popc(ms);
      ne += __popc(me);
    }
    for (int64_t t = ns + lane; t < L; t += 32) {
      tokens[b * L + t] = -1;
      starts[b * L + t] = -1;
      ends[b * L + t] = -1;
    }
    if (lane == 0) {
      lens[b] = ns;
      s_count = ns;
    }
  } else if (warp == 1 && lane == 0) {
    double sum = 0.0;
    for (int64_t t = 0; t < Lb; ++t) sum += (double)q[t];
    log_prob[b] = sum;
  }
  __syncthreads();
  const int count = s_count;
  for (int64_t k = threadIdx.x; k < L; k += 256) {
    double sum = 0.0;
    if (k < count) {
      const int64_t e = ends[b * L + k];
      for (int64_t t = starts[b * L + k]; t < e; ++t) sum += (double)q[t];
    }
    tok_lp[b * L + k] = sum;
  }
}

}  // namespace

cudaError_t launch_ctc_confidence(int32_t* pred, float* lp, const float* logits, const float2* stats, int V,
                                  const float* amax_val, const int32_t* amax_idx, const float* amax_sum, int slots,
                                  int32_t* tokens, int32_t* starts, int32_t* ends, double* token_log_probs,
                                  int32_t* lens, double* log_probs, int64_t B, int64_t L, int blank,
                                  const int32_t* lens_in, int lens_stride, cudaStream_t s, int64_t* launches) {
  if (B <= 0) return cudaSuccess;
  if (amax_val ? (!amax_idx || !amax_sum || slots <= 0) : (B * L > 0 && (!logits || !stats))) return cudaErrorInvalidValue;
  const cudaError_t e =
      amax_val ? launch_k(ctc_confidence_kernel<true>, dim3((unsigned)B), dim3(256), 0, s, pred, lp, logits, stats, V,
                          amax_val, amax_idx, amax_sum, slots, B * L, tokens, starts, ends, token_log_probs, lens,
                          log_probs, L, blank, lens_in, lens_stride)
               : launch_k(ctc_confidence_kernel<false>, dim3((unsigned)B), dim3(256), 0, s, pred, lp, logits, stats,
                          V, amax_val, amax_idx, amax_sum, 0, B * L, tokens, starts, ends, token_log_probs, lens,
                          log_probs, L, blank, lens_in, lens_stride);
  if (launches) ++*launches;
  return e;
}

cudaError_t launch_ctc_runs(const int32_t* pred, int32_t* tokens, int32_t* starts, int32_t* ends, int32_t* lens,
                            int64_t B, int64_t L, int blank, cudaStream_t s, int64_t* launches) {
  if (B <= 0) return cudaSuccess;
  ctc_runs_kernel<<<(unsigned)B, 32, 0, s>>>(pred, tokens, starts, ends, lens, L, blank);
  if (launches) ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_argmax(const float* logits, int32_t* pred, int64_t M, int V, cudaStream_t s,
                          int64_t* launches) {
  if (M <= 0) return cudaSuccess;
  const cudaError_t e = launch_k(argmax_kernel, dim3((unsigned)((M + 7) / 8)), dim3(256), 0, s, logits, pred, M, V);
  if (launches) ++*launches;
  return e;
}

cudaError_t launch_ctc_collapse(int32_t* pred, int32_t* tokens, int32_t* lens, int64_t B, int64_t L,
                                int blank, int collapse, cudaStream_t s, int64_t* launches, const int32_t* rag,
                                const float* amax_val, const int32_t* amax_idx, int slots) {
  if (B <= 0) return cudaSuccess;
  const cudaError_t e =
      amax_val ? launch_k(ctc_collapse_kernel<true>, dim3((unsigned)B), dim3(256), 0, s, pred, tokens, lens, L, blank,
                          collapse, rag, amax_val, amax_idx, slots, B * L)
               : launch_k(ctc_collapse_kernel<false>, dim3((unsigned)B), dim3(32), 0, s, pred, tokens, lens, L, blank,
                          collapse, rag, amax_val, amax_idx, 0, B * L);
  if (launches) ++*launches;
  return e;
}

}  // namespace vasr
