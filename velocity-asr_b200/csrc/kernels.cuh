// kernels.cuh — host-side launchers of every kernel in libvasr.  Each returns the CUDA
// error of its launch.  `launches` (may be NULL) is incremented once per kernel launched.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace vasr {

// ---------------------------------------------------------------- dense projections -----
// C[m, n] = epi( sum_k A[m, k] * W[n, k] ), A rows K-contiguous, W (N, K) as nn.Linear stores it.
// Row m of A lives at A + (m / rows_per_batch) * batch_stride + (m % rows_per_batch) * lda,
// which lets a strided / overlapping view (conv frames, STFT frames) be used without im2col.
// Epilogue, in order: + bias[n]; FakeQuantize with per-column (q_scale[n], q_zp[n]) when given (config 5);
// act on columns n >= act_from; + pos-enc (time table row
// m % pe_rows for n < pe_half, learned freq vector for n >= pe_half); + resid[m, n].
struct GemmArgs {
  const float* A = nullptr;
  int64_t lda = 0;
  int64_t rows_per_batch = 0;  // 0 -> plain matrix
  int64_t batch_stride = 0;
  const float* W = nullptr;
  const float* W_split = nullptr;  // [rna_tf32(W) | rna_tf32(W - hi)], 2*N*K floats (launch_split_tf32); tensor-core path only
  const float* bias = nullptr;
  const float* q_scale = nullptr;  // (N) device; with q_zp: output FakeQuantize per column (scale <= 0: none)
  const float* q_zp = nullptr;
  float* C = nullptr;
  int64_t ldc = 0;
  int64_t M = 0, N = 0, K = 0;
  int act = 0;
  int act_from = 0;
  const float* resid = nullptr;
  int64_t ldr = 0;
  // LayerNorm folded into the projection (tensor-core kernel): A holds the LayerNorm's INPUT rows (K = the
  // normalised width), W is W diag(gamma), bias is b + W beta, ln_s[n] = sum_k W'[n, k]; ln_stats: (M, 2) scratch
  const float* ln_s = nullptr;
  float* ln_stats = nullptr;
  float ln_eps = 1e-5f;
  // greedy decode: instead of C, per row and slot p = 2 * (n / 128) + half the (max, first argmax) of the columns
  // the slot covers, at amax_val / amax_idx[p * M + m]; launch_ctc_collapse takes them (argmax_slots(N) slots)
  float* amax_val = nullptr;
  int32_t* amax_idx = nullptr;
  // GatedFusion: W rows permuted by gate_perm_row (N = 3 C): C[m, c] = s l + (1 - s) t, s = sigmoid(gate), C is (M, C)
  int gate = 0;
  const float* pe_time = nullptr;  // (>= pe_rows, pe_half)
  const float* pe_freq = nullptr;  // (N - pe_half)
  int pe_half = 0;
  int64_t pe_rows = 0;
};
// CUDA-core fp32 kernel behind vasr_linear (a general-purpose op for views the tensor-core kernel cannot take,
// e.g. K % 4 != 0); the model's launch sequence never uses it.
cudaError_t launch_gemm(const GemmArgs& g, cudaStream_t s, int64_t* launches);
// tcgen05 / TMEM / TMA path with 3xTF32 split accumulation (gemm_tc.cu); needs g.W_split.  Returns
// cudaErrorNotSupported when a tensor map cannot be encoded for this view.
cudaError_t launch_gemm_tc(const GemmArgs& g, int num_sms, cudaStream_t s, int64_t* launches);
// The template instantiation a launch_gemm_tc call launched (family 1 = gemm_tc_kernel, 2 = gemm_tc2_kernel; tn, act,
// pe, resid, quant, wres, epi = its template arguments).  Each launch site sets it; the projection tests read it.
struct TcVariant {
  int family, tn, act, pe, resid, quant, wres, epi;
};
extern thread_local const TcVariant* tc_last_variant;
// hl[0..n) = rna_tf32(w), hl[n..2n) = rna_tf32(w - hl[0..n)): the weight operand of launch_gemm_tc.
cudaError_t launch_split_tf32(const float* w, float* hl, int64_t n, cudaStream_t s);
extern long long* g_trace;   // debug: device buffer (5 x 128 clock64 slots) CTA 0 of the projection kernel writes

// ---------------------------------------------------------------- quantisation (config 5) ---
// mm[0] = min, mm[1] = max over x[m, c0 .. c0+nc) for m < M (row stride ldx).  Deterministic (one CTA).
cudaError_t launch_minmax(const float* x, int64_t ldx, int64_t M, int c0, int nc, float* mm, cudaStream_t s,
                          int64_t* launches);
// FakeQuantize._update_scale_zp for an asymmetric per-tensor uint8 node (quantize.py:116-121):
// scale = max((max - min) / 255, 1e-10), zp = 0 - min / scale, written to q_scale/q_zp[c0 .. c0+nc).
cudaError_t launch_set_qparams(const float* mm, float* q_scale, float* q_zp, int c0, int nc, cudaStream_t s,
                               int64_t* launches);

// ---------------------------------------------------------------- normalisation / conv ---
// y[m, :] = LayerNorm(x[m, :]) * gamma + beta over C channels (eps 1e-5, biased variance).
cudaError_t launch_layer_norm(const float* x, int64_t ldx, float* y, int64_t ldy, const float* gamma,
                              const float* beta, int64_t M, int C, cudaStream_t s, int64_t* launches);
// u = causal depthwise conv_k( LayerNorm(x) ) + bias on (B, L, C); zero left padding is
// applied to the LayerNorm output (ssm.py:408-414).  w: (C, k) row-major.  A warp takes run_len consecutive
// tokens (0: the launcher's rule, which fills whole waves of the GPU); the run length used goes to *run_len_used.
cudaError_t launch_ln_dwconv(const float* x, float* u, const float* gamma, const float* beta,
                             const float* w, const float* bias, int64_t B, int64_t L, int C, int k,
                             cudaStream_t s, int64_t* launches, int run_len = 0, int* run_len_used = nullptr);

// ---------------------------------------------------------------- selective scan --------
struct ScanArgs {
  const float* x = nullptr;   int64_t ldx = 0;
  const float* dt = nullptr;  int64_t lddt = 0;
  const float* z = nullptr;   int64_t ldz = 0;   // NULL -> no gate
  const float* Bm = nullptr;  int64_t ldb = 0;
  const float* Cm = nullptr;  int64_t ldc = 0;
  const float* A = nullptr;                       // (N), negative
  const float* D = nullptr;                       // (Di) or NULL
  float* y = nullptr;         int64_t ldy = 0;
  int64_t B = 0, L = 0;
  int Di = 0, N = 0;
  int parallel_quirk = 0;     // 0: true recurrence (sequential/mamba); 1: reference 'parallel'
  int structured_a = 0;       // A[n] == -(n+1): powers of exp(-dt) instead of one exp per state
  int num_sms = 0;            // 0 -> 148
};
cudaError_t launch_selective_scan(const ScanArgs& a, cudaStream_t s, int64_t* launches);

// ---------------------------------------------------------------- ragged batches ---------
// A batch whose utterances have different lengths is stored padded to the longest; `rag` (device,
// B x RAG_STRIDE int32) holds what each utterance really has.  Everything along time is causal or
// per-token except the five places that take `rag`: the reflect padding and frame count of the mel,
// its statistics, the zero frames after the end, both adaptive poolings, the number of attention keys
// and the decode length.  NULL = every utterance spans the full rows.
enum { RAG_S = 0, RAG_T = 1, RAG_L = 2, RAG_K1 = 3, RAG_K2 = 4, RAG_STRIDE = 8 };

// ---------------------------------------------------------------- log-mel front end -----
// One pass PCM (B, S) -> raw (B, T, n_mels) = log(mel power + 1e-10): reflect padding by index, window,
// 400-point FFT, power, band-sparse filterbank (weights fb_w[fb_off[j] .. fb_off[j+1]) on frequency bins
// fb_lo[j] ...), log.  win: 400 taps; tw: 400 x (cos, -sin)(2 pi m / 400).  part (B, mel_fft_blocks(T),
// n_mels, 2) doubles receives per-CTA (mean, M2) partials for launch_mel_finish (NULL to skip).
int64_t mel_fft_blocks(int64_t T);
cudaError_t launch_mel_fft(const float* pcm, float* raw, double* part, int64_t B, int64_t S, int64_t T, int n_mels,
                           const int* fb_lo, const int* fb_off, const float* fb_w, const float* win,
                           const float* tw, cudaStream_t s, int64_t* launches, const int32_t* rag = nullptr);
// out[b, t + front, j] = (raw[b,t,j] - mean[b,j]) * rstd[b,j]; out has frames_per_utt rows per utterance, rows
// outside [front, front + T) are zeroed.  The statistics — per (b, j) the mean and 1 / (unbiased std + 1e-10) over
// the T frames — come from `part` (the partials of launch_mel_fft, merged inside the kernel); without it the kernel
// is a plain copy.
cudaError_t launch_mel_finish(const float* raw, float* out, int64_t B,
                              int64_t T, int n_mels, int64_t frames_per_utt, int front, cudaStream_t s,
                              int64_t* launches, const int32_t* rag = nullptr, const double* part = nullptr);

// ---------------------------------------------------------------- global context --------
// out[b, i, :] = mean_t x[b, floor(iL/K) .. ceil((i+1)L/K), :]   (attention.py:71-73)
// ragged: the input length is rag[b][f_in] and the output count rag[b][f_out] (rows past it are zeroed)
cudaError_t launch_adaptive_pool(const float* x, int64_t ldx, float* out, int64_t B, int64_t L, int64_t K,
                                 int C, cudaStream_t s, int64_t* launches, const int32_t* rag = nullptr,
                                 int f_in = 0, int f_out = 0);
// q (B*L, heads*hd) stride ldq; kv (B*Kk, 2*heads*hd): [k | v]; o (B*L, heads*hd) stride ldo.
cudaError_t launch_attention(const float* q, int64_t ldq, const float* kv, float* o, int64_t ldo, int64_t B,
                             int64_t L, int64_t Kk, int heads, int hd, cudaStream_t s, int64_t* launches,
                             const int32_t* rag = nullptr);
// f3 (M, 3C): [gate_logit | local_t | global_t] -> out (M, C) = s*lt + (1-s)*gt, s = sigmoid(gate).
cudaError_t launch_gate_mix(const float* f3, float* out, int64_t M, int C, cudaStream_t s, int64_t* launches);

// ---------------------------------------------------------------- CTC greedy ------------
cudaError_t launch_argmax(const float* logits, int32_t* pred, int64_t M, int V, cudaStream_t s,
                          int64_t* launches);
// tokens / starts / ends (B, L) left-packed: run starts of equal non-blank predictions, with [start, end) frames
cudaError_t launch_ctc_runs(const int32_t* pred, int32_t* tokens, int32_t* starts, int32_t* ends, int32_t* lens,
                            int64_t B, int64_t L, int blank, cudaStream_t s, int64_t* launches);
// amax_val / amax_idx (slots x B*L): each frame's prediction is first taken from the CTC-head projection's argmax
// partials (GemmArgs::amax_val) and written to `pred`
inline int argmax_slots(int64_t N) { return (int)(2 * ((N + 127) / 128)); }
cudaError_t launch_ctc_collapse(int32_t* pred, int32_t* tokens, int32_t* lens, int64_t B, int64_t L,
                                int blank, int collapse, cudaStream_t s, int64_t* launches,
                                const int32_t* rag = nullptr, const float* amax_val = nullptr,
                                const int32_t* amax_idx = nullptr, int slots = 0);

// ---------------------------------------------------------------- CTC prefix beam search
// per (utterance, frame) row: stats = (max, log sum exp(x - max)); top_tok (M, K) = the K best non-blank
// tokens by log-prob, ties to the lower id, -1 padded.  M = B * L.  lens (optional, B entries at lens[b *
// lens_stride], e.g. the RAG_L column of a ragged dims buffer): rows b * L + t with t >= lens[b] are skipped.
cudaError_t launch_beam_rows(const float* logits, float2* stats, int32_t* top_tok, int64_t M, int V, int K,
                             int blank, int64_t L, const int32_t* lens, int lens_stride, cudaStream_t s,
                             int64_t* launches);
// trie: 3 x (B, trie_cap) int32 (parent | token | depth), trie_cap >= 1 + L * W.  out_tokens (B, W, L),
// out_lens (B, W) (-1 = no such beam), out_scores (B, W) fp64, best first.  lens as in launch_beam_rows:
// utterance b is searched over its first lens[b] rows (NULL: all L); its token rows are -1 past each beam's length.
cudaError_t launch_beam_search(const float* logits, const float2* stats, const int32_t* top_tok, int K, int64_t B,
                               int64_t L, const int32_t* lens, int lens_stride, int V, int W, int blank,
                               int32_t* trie, int64_t trie_cap, int32_t* out_tokens, int32_t* out_lens,
                               double* out_scores, cudaStream_t s, int64_t* launches);

// ---------------------------------------------------------------- CTC forced alignment / log-likelihood
// One CTA per utterance over the 2U+1 states of its target (align.cu).  ctc_align_layout gives the CTA size and the
// states per thread for the longest target U (viterbi: E a multiple of 16, so a backpointer word has one writer);
// ctc_align_smem the dynamic shared memory, with or without the scores (fp64, E * threads of them) in it.
int64_t ctc_align_words(int64_t U);   // backpointer words per (utterance, frame): ceil((2U + 1) / 16)
void ctc_align_layout(int64_t U, bool viterbi, int* threads, int* E);
size_t ctc_align_smem(int threads, int E, bool delta_in_smem);
// stats: launch_beam_rows' (max, log sum exp) per row, or NULL when the logits are log-probs.  lens as in
// launch_beam_rows.  targets (B, U_max) with target_lens (B), device.  delta_g: NULL (scores in shared memory) or
// (B, E * threads) doubles.  bp != NULL: Viterbi, with bp (B, L, words) scratch, out_labels / out_lp (B, L) and the
// path score in out_score (B); bp == NULL: the log-likelihood in out_score.
cudaError_t launch_ctc_align(const float* logits, const float2* stats, int64_t B, int64_t L, int V, int blank,
                             const int32_t* lens, int lens_stride, const int32_t* targets, int64_t U_max,
                             const int32_t* target_lens, int threads, int E, double* delta_g, uint32_t* bp,
                             int64_t words, int32_t* out_labels, float* out_lp, double* out_score, cudaStream_t s);

}  // namespace vasr
