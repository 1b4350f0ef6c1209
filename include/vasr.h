/* vasr.h — C ABI of libvasr.so, the B200 (sm_100a) inference path for VELOCITY-ASR v2.
 *
 * The reference (shaderko/velocity-asr) is pure Python/PyTorch and has no FFI of its own
 * (SURVEY.md section 8b).  Its two seams are the package API (velocity_asr/__init__.py:95-145)
 * and the scan_mode switch (velocity_asr/ssm.py:119-126).  Each entry point below replaces
 * one reference callable; the Python package in velocity-asr_b200/velocity_asr binds them
 * with ctypes (see INTEGRATION.md) and keeps the reference's names and argument meaning.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types.  `*_dev` pointers are device memory on
 *     the handle's GPU, `*_host` pointers are host memory.  All tensors are contiguous fp32
 *     in the reference's own layouts (channels-last: (B, T, C)).
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls are
 *     asynchronous with respect to the host unless the name ends in `_host`.
 *   - every function returns VASR_OK or an error code; vasr_last_error() gives the text for
 *     the calling thread.  There is no CPU fallback: without a CUDA device every compute
 *     entry point fails with VASR_ERR_CUDA.
 *   - the caller owns all buffers it passes; the handle owns weights and workspace.  The
 *     workspace grows on first use of a larger (B, S) and is then reused: no allocation on
 *     the hot path after warm-up.  One handle per GPU per process; calls on one handle must
 *     not overlap.
 */
#ifndef VASR_H_
#define VASR_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vasr_handle vasr_handle;

enum {
  VASR_OK = 0,
  VASR_ERR_INVALID = 1,     /* bad argument / unknown name -> ValueError (ssm.py:126)            */
  VASR_ERR_SHAPE = 2,       /* shape the model cannot take -> RuntimeError (model.py:125)        */
  VASR_ERR_CUDA = 3,        /* CUDA runtime / no device                                          */
  VASR_ERR_STATE = 4,       /* weights missing or not committed                                  */
  VASR_ERR_UNSUPPORTED = 5  /* configuration outside what the kernels are built for              */
};

enum { VASR_SCAN_SEQUENTIAL = 0, VASR_SCAN_PARALLEL = 1, VASR_SCAN_MAMBA = 2 };

/* Mirrors VelocityASRConfig (velocity_asr/model.py:23-68); dropout / checkpointing /
 * use_compile have no meaning for inference and are not carried. */
typedef struct vasr_config {
  int32_t mel_bins;              /* 80  */
  int32_t d_model;               /* 192 */
  int32_t ssm_layers;            /* 8   */
  int32_t ssm_state_dim;         /* 64  */
  int32_t ssm_expand_ratio;      /* 2   */
  int32_t ssm_kernel_size;       /* 4   */
  int32_t global_ssm_layers;     /* 2   */
  int32_t global_ssm_state_dim;  /* 32  */
  int32_t attention_heads;       /* 4   */
  int32_t attention_dim;         /* 48  */
  int32_t vocab_size;            /* 1000 */
  int32_t scan_mode;             /* VASR_SCAN_*; the reference default is PARALLEL (model.py:60) */
} vasr_config;

const char* vasr_last_error(void);
const char* vasr_version(void);

/* ---- handle and weights: VELOCITYASR.__init__ / load_state_dict (model.py:255-299, 416-431) */
int vasr_create(const vasr_config* cfg, int device, vasr_handle** out);
void vasr_destroy(vasr_handle* h);
/* One tensor of the reference state_dict, by its reference key (the 208 names of SURVEY.md
 * section 8b), fp32, host memory, numel elements.  Two extra optional keys override the
 * built-in front-end tables: "frontend.mel_filterbank" (n_mels x 201) and "frontend.window"
 * (400).  Unknown keys -> VASR_ERR_INVALID. */
int vasr_set_weight(vasr_handle* h, const char* name, const float* host, int64_t numel);
/* Packs the tensors into kernel layouts; fails with VASR_ERR_STATE naming the first missing key. */
int vasr_commit_weights(vasr_handle* h);

/* ---- shape helpers: audio.py:104-112 (center=False after reflect pad), model.py:370-383 */
int64_t vasr_num_frames(int64_t samples);   /* 1 + samples / 160                 */
int64_t vasr_num_tokens(int64_t frames);    /* (frames + 1) / 2                  */

/* ---- compute_mel_spectrogram (velocity_asr/audio.py:65-143)
 * pcm (B, S) -> mel (B, T, n_mels), T = vasr_num_frames(S).  S must be > 200 (reflect pad).  n_mels is the
 * handle's mel_bins, any value in [1, 128]; the model's projections need 3 * mel_bins to be a multiple of 16,
 * which vasr_commit_weights checks. */
int vasr_log_mel(vasr_handle* h, const float* pcm_dev, int64_t B, int64_t S, int normalize,
                 float* mel_dev, void* stream);

/* ---- VELOCITYASR.forward (velocity_asr/model.py:333-368)
 * mel (B, T, mel_bins) -> logits (B, L, vocab), L = vasr_num_tokens(T).  The three feature
 * pointers are the return_features dict ('temporal_binding', 'local_features',
 * 'fused_features'), each (B, L, d_model); pass NULL to skip. */
int vasr_forward(vasr_handle* h, const float* mel_dev, int64_t B, int64_t T, float* logits_dev,
                 float* feat_tb_dev, float* feat_local_dev, float* feat_fused_dev, void* stream);

/* ---- module-level seams used by the parity tests (reference classes in __all__) ---------- */
/* SSMBlock.forward (ssm.py:404-427).  stack 0 = local_ssm.layers[layer], 1 =
 * global_context.global_ssm.layers[layer]; scan_mode < 0 = the mode the reference would use
 * (config scan_mode for local, PARALLEL for global, ssm.py:529-538). */
int vasr_ssm_block(vasr_handle* h, int stack, int layer, int scan_mode, const float* x_dev,
                   int64_t B, int64_t L, float* out_dev, void* stream);
/* HierarchicalGlobalContext.forward (attention.py:283-319): (B, L, d_model) -> same. */
int vasr_global_context(vasr_handle* h, const float* local_dev, int64_t B, int64_t L,
                        float* out_dev, void* stream);
/* CTCOutputHead.forward (model.py:229-239): (B, L, d_model) -> (B, L, vocab). */
int vasr_ctc_head(vasr_handle* h, const float* x_dev, int64_t B, int64_t L, float* logits_dev,
                  void* stream);

/* ---- the scan operator: SelectiveSSM._sequential_scan / _parallel_scan / _mamba_scan
 * (ssm.py:134-337).  x, dt: (B, L, Di) with row strides ldx, lddt; Bm, Cm: (B, L, N) with row
 * strides ldb, ldc; A: (N), D: (Di) or NULL (no skip term); z: (B, L, Di) stride ldz or NULL
 * (when given, y is multiplied by silu(z), ssm.py:129); y: (B, L, Di) stride ldy.
 * N in {16, 32, 64}.  All device pointers.  No handle: the operator is stateless. */
int vasr_selective_scan(const float* x, int64_t ldx, const float* dt, int64_t lddt, const float* A,
                        const float* Bm, int64_t ldb, const float* Cm, int64_t ldc, const float* D,
                        const float* z, int64_t ldz, float* y, int64_t ldy, int64_t B, int64_t L,
                        int64_t Di, int64_t N, int scan_mode, void* stream);

/* ---- ctc_greedy_decode (velocity_asr/decode.py:27-71)
 * logits (B, L, V) -> tokens (B, L) int32 left-packed, lens (B) int32.  argmax ties -> lowest
 * index; blanks dropped; repeats collapsed when collapse != 0; a blank resets the repeat state. */
int vasr_ctc_greedy(const float* logits_dev, int64_t B, int64_t L, int64_t V, int blank, int collapse,
                    int32_t* tokens_dev, int32_t* lens_dev, void* stream);

/* ---- ctc_greedy_decode_with_timestamps (velocity_asr/decode.py:74-125)
 * As above with repeats collapsed, plus per token the [start, end) frame range of its run of equal
 * predictions: tokens / starts / ends (B, L) int32 left-packed, lens (B). */
int vasr_ctc_greedy_timestamps(const float* logits_dev, int64_t B, int64_t L, int64_t V, int blank,
                               int32_t* tokens_dev, int32_t* starts_dev, int32_t* ends_dev, int32_t* lens_dev,
                               void* stream);

/* ---- ragged batches (the reference's collator pads with zeros and never masks, data.py:145-203, so an
 * utterance's transcript depends on its batch mates; these entry points take the true lengths instead)
 * pcm (B, S) holds utterance b in its first sample_lens[b] samples (200 < len <= S; the rest is ignored).
 * Each utterance is processed exactly as if it were alone: reflect padding, frame count and mel statistics from
 * its own length, zero frames after its end, pooling windows and attention keys from its own token count, decode
 * over its own tokens.  tokens (B, L) / lens (B) as vasr_transcribe, L = vasr_num_tokens(vasr_num_frames(S)).
 * sample_lens / frame_lens are HOST arrays.  vasr_forward_ragged: mel (B, T, n_mels) with frame_lens[b] valid
 * frames (1 <= len <= T); logits rows at or past an utterance's own token count are padding. */
int vasr_transcribe_ragged(vasr_handle* h, const float* pcm_dev, const int32_t* sample_lens_host, int64_t B,
                           int64_t S, int32_t* tokens_dev, int32_t* lens_dev, void* stream);
int vasr_transcribe_ragged_host(vasr_handle* h, const float* pcm_host, const int32_t* sample_lens_host, int64_t B,
                                int64_t S, int32_t* tokens_host, int32_t* lens_host);
int vasr_forward_ragged(vasr_handle* h, const float* mel_dev, const int32_t* frame_lens_host, int64_t B, int64_t T,
                        float* logits_dev, void* stream);

/* ---- ctc_beam_search (velocity_asr/decode.py:128-217), lm_scorer = None
 * Prefix beam search with the reference's max-merge rule, fp64 scores and insertion-order tie-breaks.
 * tokens (B, beam_width, L) int32 (-1 padded), lens (B, beam_width) int32 (-1 where the utterance has fewer
 * beams), scores (B, beam_width) fp64, best beam first.  1 <= beam_width <= 32. */
int vasr_ctc_beam_search(const float* logits_dev, int64_t B, int64_t L, int64_t V, int beam_width, int blank,
                         int32_t* tokens_dev, int32_t* lens_dev, double* scores_dev, void* stream);

/* ---- n-gram language model over token ids (ARPA), fused into the prefix beam search
 * lm(prefix, tok), natural log: the history is ("<s>",) + prefix cut to its last order-1 items; P(w | h) = p(h w)
 * when listed, else bow(h) + P(w | h[1:]) (bow of an unlisted context = 0); a token without a unigram takes the
 * <unk> unigram.  Every ARPA value (log10) is parsed as fp64, times ln 10 in fp64, rounded once to fp32; the
 * back-off sum is fp64 (the listed entry found, then the back-off weights from the shortest context outward),
 * rounded to fp32.  An ARPA word maps to the vocabulary entry with the same string, <space> to " "; n-grams with a
 * word outside the vocabulary are dropped, <s> is kept as a context, </s> is unused, the blank is never scored. */
typedef struct vasr_lm vasr_lm;
/* Parses the ARPA file at `path` for a vocabulary of V NUL-terminated UTF-8 strings and uploads its tables to
 * `device` (< 0: the calling thread's current device).  Malformed files (bad header, section counts that differ
 * from \data\, an unparsable number, no \end\), an order above 8, and a non-blank token with no unigram in a file
 * without <unk> fail with VASR_ERR_INVALID and a message naming the line, before any device call. */
int vasr_lm_create_arpa(const char* path, const char* const* vocab, int64_t V, int blank, int device, vasr_lm** out);
void vasr_lm_destroy(vasr_lm* lm);
int vasr_lm_order(const vasr_lm* lm);
/* out[i] = lm(prefix_i, tokens[i]) fp32, n rows.  prefixes (n, max(order-1, 1)) int32 holds the last
 * min(len_i, order-1) tokens of prefix i right-aligned (newest last); prefix_lens (n) its true length, so a prefix
 * shorter than order-1 starts at <s>.  All device pointers on the LM's device; a token outside [0, V) gives NaN. */
int vasr_lm_log_prob(const vasr_lm* lm, const int32_t* prefixes_dev, const int32_t* prefix_lens_dev, int64_t n,
                     const int32_t* tokens_dev, float* out_dev, void* stream);
/* vasr_ctc_beam_search with shallow fusion: an offer that extends a prefix by tok scores
 * (score + log_prob[tok]) + lm_weight * lm(prefix, tok) in fp64; blank and repeat offers are unchanged.  Outputs as
 * vasr_ctc_beam_search, scores are the fused ones.  The LM must be built for this V and blank, and logits_dev must be
 * device memory on the LM's device (else VASR_ERR_INVALID); lm_weight finite.  1 <= beam_width <= 32. */
int vasr_ctc_beam_search_lm(const float* logits_dev, int64_t B, int64_t L, int64_t V, int beam_width, int blank,
                            const vasr_lm* lm, double lm_weight, int32_t* tokens_dev, int32_t* lens_dev,
                            double* scores_dev, void* stream);

/* ---- word-level n-gram LM over a character vocabulary, fused into the prefix beam search
 * The LM above over the file's own words: word id = index in the unigram section (first occurrence, <s> excluded),
 * <s> is the context symbol, </s> and <unk> are ordinary words; lm(h, w) is the rule above over word ids.
 * d = the vocabulary entry `delimiter` (the first one).  Spelling: a word's characters (UTF-8 code points), one
 * token each, the first vocabulary entry with that one-character string, which must be neither the blank nor d;
 * a word that cannot be spelled stays in the LM but not in the lexicon = the spellable unigram words other than
 * <s>, </s>, <unk>.
 * A prefix P (collapsed token ids) splits at each d into runs: the non-empty runs before the last d are its words
 * w_1 .. w_k, the tokens after the last d its pending run u (possibly empty); word(run) = the lexicon word spelled
 * by the run, else <unk>;
 * h(P) = (<s>, word(w_1), ..., word(w_k)) cut to its last order-1 items.
 * Offers from hypothesis (P, s, last) at a frame with fp32 log-softmax lp, summed in fp64 in exactly this order:
 *   blank, repeat of last: P kept, s + lp[tok], no LM term (as vasr_ctc_beam_search);
 *   d (d != last): u empty -> P+d, s + lp[d]; else ((s + lp[d]) + lm_weight * lm(h(P), word(u))) + word_score;
 *     constrained: not offered when u is non-empty and not a lexicon word;
 *   any other t: P+t, s + lp[t]; constrained: offered only when u+t is a prefix of a lexicon word's spelling.
 *   Max-merge, first offer wins a tie, the stable top beam_width: as vasr_ctc_beam_search.
 * End of utterance, per surviving hypothesis, in order: (1) u non-empty: constrained and u not a lexicon word ->
 * dropped (len -1, as a missing beam); else s = (s + lm_weight * lm(h, word(u))) + word_score and word(u) joins the
 * history; (2) s += lm_weight * lm(h', </s>) (</s> absent from the file: <unk>); (3) a stable sort by s, descending.
 * L = 0 gives the empty beam with lm_weight * lm((<s>), </s>). */
/* Parses a word ARPA file and builds the lexicon for a vocabulary of V strings; constrained != 0 limits hypotheses
 * to lexicon words.  VASR_ERR_INVALID, before any device call, for: a delimiter missing from the vocabulary or equal
 * to the blank, the malformed files of vasr_lm_create_arpa (naming the line), lexicon-free mode without <unk>, a
 * file with neither </s> nor <unk>, constrained mode with an empty lexicon.  vasr_lm_order, vasr_lm_destroy and
 * vasr_lm_log_prob (over word ids) take the result. */
int vasr_lm_create_word_arpa(const char* path, const char* const* vocab, int64_t V, int blank, const char* delimiter,
                             int constrained, int device, vasr_lm** out);
/* ids_host[i] = the word id of words[i]; a string that is not a word of the LM maps to <unk> (fails without one). */
int vasr_lm_word_ids(const vasr_lm* lm, const char* const* words, int64_t n, int32_t* ids_host);
/* The lexicon size of a word LM, -1 for a token LM. */
int64_t vasr_lm_lexicon_size(const vasr_lm* lm);
/* The search with a word LM, outputs as vasr_ctc_beam_search_lm; returned scores are the final ones (after the end
 * of utterance).  lm_weight finite and >= 0, word_score finite.  A token LM here, or a word LM given to
 * vasr_ctc_beam_search_lm, fails with VASR_ERR_INVALID. */
int vasr_ctc_beam_search_word_lm(const float* logits_dev, int64_t B, int64_t L, int64_t V, int beam_width, int blank,
                                 const vasr_lm* lm, double lm_weight, double word_score, int32_t* tokens_dev,
                                 int32_t* lens_dev, double* scores_dev, void* stream);

/* ---- the prefix beam search over a ragged batch, with or without an LM
 * lm == NULL runs the rule of vasr_ctc_beam_search (lm_weight and word_score are not used); a token LM the rule of
 * vasr_ctc_beam_search_lm (word_score must be 0); a word LM the rule of vasr_ctc_beam_search_word_lm.  Argument
 * checks, messages and the LM's device and vocabulary requirements are those of the matching entry point.
 * row_lens_host: B frame counts, a HOST array that may be reused as soon as the call returns, or NULL (every
 * utterance has L frames).  Each 0 <= row_lens[b] <= L, else VASR_ERR_SHAPE before any device work.  Utterance b is
 * searched over rows b*L + [0, row_lens[b]) of logits (B, L, V); the rows after them are never read, so whatever
 * they hold (NaN included) does not matter.  A word LM's end-of-utterance step follows the utterance's last frame.
 * Outputs keep the shapes of vasr_ctc_beam_search: tokens (B, beam_width, L), -1 past each beam's length.
 * Contract: utterance b gets bit for bit the tokens, lens and fp64 scores that the matching unragged entry point
 * gives for logits[b : b+1, : row_lens[b]] alone.  row_lens[b] = 0 gives the L = 0 result: the single empty beam
 * with score 0, or lm_weight * lm((<s>), </s>) under a word LM. */
int vasr_ctc_beam_search_ragged(const float* logits_dev, const int32_t* row_lens_host, int64_t B, int64_t L,
                                int64_t V, int beam_width, int blank, const vasr_lm* lm, double lm_weight,
                                double word_score, int32_t* tokens_dev, int32_t* lens_dev, double* scores_dev,
                                void* stream);

/* ---- transcribe with the beam search: PCM -> log-mel -> model -> logits -> prefix beam search, one call.
 * pcm (B, S); sample_lens_host (optional, HOST): a ragged batch as vasr_transcribe_ragged (200 < len <= S, else
 * VASR_ERR_SHAPE).  L = vasr_num_tokens(vasr_num_frames(S)), blank = 0.  Outputs as vasr_ctc_beam_search_ragged:
 * tokens (B, beam_width, L), lens (B, beam_width), scores (B, beam_width) fp64.  lm: NULL, a token LM or a word LM,
 * rules and checks as vasr_ctc_beam_search_ragged; it must live on the handle's device and be built for vocab_size
 * and blank 0, else VASR_ERR_INVALID before any device work.  The CTC head writes the logits (as vasr_forward) into
 * the handle's workspace, which grows by B * L * vocab_size floats for these calls only.
 * Contract: utterance b gets bit for bit what vasr_ctc_beam_search_ragged gives on the logits vasr_forward produces
 * for that utterance alone (its first sample_lens[b] samples, or all S).  The _host variant takes host PCM, returns
 * host results and synchronises once at the end. */
int vasr_transcribe_beam(vasr_handle* h, const float* pcm_dev, const int32_t* sample_lens_host, int64_t B, int64_t S,
                         int beam_width, const vasr_lm* lm, double lm_weight, double word_score, int32_t* tokens_dev,
                         int32_t* lens_dev, double* scores_dev, void* stream);
int vasr_transcribe_beam_host(vasr_handle* h, const float* pcm_host, const int32_t* sample_lens_host, int64_t B,
                              int64_t S, int beam_width, const vasr_lm* lm, double lm_weight, double word_score,
                              int32_t* tokens_host, int32_t* lens_host, double* scores_host);

/* ---- CTC forced alignment and transcript log-likelihood
 * Inputs: logits (B, L, V), utterance b over its first row_lens[b] frames; a target y = targets[b, :target_lens[b]]
 * of length U; blank.  Per-frame log-probs lp[t][v]: by default the beam search's fp32 table
 * (x - max) - log sum exp(x - max), from the statistics of beam_rows_kernel; with log_probs != 0 the inputs already
 * are log-probs and are read as they are.
 * States are the usual CTC expansion blank, y0, blank, y1, ..., blank: 2U + 1 states with label(s).  From s-1 any
 * state may be entered; from s-2 only when label(s) != blank and label(s) != label(s-2).  All sums are fp64 of fp32
 * lp values, added in time order.
 * Viterbi (vasr_ctc_align): delta[0][0] = lp[0][blank], delta[0][1] = lp[0][y0], every other state at frame 0 is
 * -inf; for t >= 1 delta[t][s] = max(delta[t-1][s], delta[t-1][s-1], delta[t-1][s-2]) + lp[t][label(s)].  Inside the
 * max the first candidate, in the order stay, s-1, s-2, that has the strictly greatest value wins.  The final state
 * is 2U-1 (last token) or 2U (trailing blank); on a tie the last-token state wins.  Outputs: frame_labels (B, L) int32,
 * the token id of the state the best path occupies at each frame, blank included; frame_log_probs (B, L) fp32, lp at
 * that frame and label; scores (B) fp64, the path score.  Equal neighbouring targets are always separated by a blank,
 * so frame labels identify target positions: token k spans [first frame in state 2k+1, last frame + 1), the units and
 * the half-open convention of vasr_ctc_greedy_timestamps.
 * Log-likelihood (vasr_ctc_log_likelihood): the same lattice with the max replaced by a log-add in fp64: with m the
 * largest present term, m + log sum exp(x_i - m), and -inf when every term is -inf; the end is the log-add of the
 * two final states.  The result equals -ctc_loss(reduction="none") of that utterance.
 * Edge cases: U = 0 is the all-blank path (with row_lens[b] = 0 as well the score is 0).  A target that cannot fit
 * (row_lens[b] < U + the number of equal neighbouring targets, row_lens[b] = 0 < U included) gets score -inf, and its
 * frames label -1 and log-prob 0.  Frames at or past row_lens[b] are never read, so NaN padding cannot matter; they
 * also get label -1 and log-prob 0.
 * Contract: utterance b gets bit for bit what the same call gives on logits[b:b+1, :row_lens[b]] with targets[b:b+1].
 * row_lens_host (B, or NULL: every utterance has L frames), targets_host (B, U_max) and target_lens_host (B) are HOST
 * arrays, copied before the call returns.  Checks, all before any device call: VASR_ERR_INVALID for a null pointer,
 * blank outside [0, V), or a target id outside [0, V) or equal to blank (only the first target_lens[b] entries of a
 * row are read); VASR_ERR_SHAPE for row_lens[b] outside [0, L] or target_lens[b] outside [0, U_max].
 * Device scratch, allocated stream-ordered per call, with U = the largest target_lens[b]: the Viterbi backpointers,
 * B * L * ceil((2U + 1) / 16) * 4 bytes (2 bits per state and frame); B * L * 8 bytes of row statistics unless
 * log_probs; and when the 2U + 1 fp64 scores of an utterance do not fit the shared memory of one CTA (U above about
 * 12,000 on a B200) about B * (2U + 1) * 8 bytes more. */
int vasr_ctc_align(const float* logits_dev, const int32_t* row_lens_host, int64_t B, int64_t L, int64_t V, int blank,
                   int log_probs, const int32_t* targets_host, const int32_t* target_lens_host, int64_t U_max,
                   int32_t* frame_labels_dev, float* frame_log_probs_dev, double* scores_dev, void* stream);
/* The same inputs; ll (B) fp64 is the only output. */
int vasr_ctc_log_likelihood(const float* logits_dev, const int32_t* row_lens_host, int64_t B, int64_t L, int64_t V,
                            int blank, int log_probs, const int32_t* targets_host, const int32_t* target_lens_host,
                            int64_t U_max, double* ll_dev, void* stream);
/* PCM -> forced alignment in one call: the sequence of vasr_transcribe_beam (log-mel, model, the CTC head writing
 * logits into the workspace, blank 0, a ragged batch by sample_lens_host) with vasr_ctc_align in place of the search.
 * L = vasr_num_tokens(vasr_num_frames(S)); outputs as vasr_ctc_align.  Works for the fp32 and the FakeQuantize model.
 * Contract: utterance b gets bit for bit what vasr_ctc_align gives on the logits vasr_forward produces for that
 * utterance alone (its first sample_lens[b] samples, or all S). */
int vasr_align(vasr_handle* h, const float* pcm_dev, const int32_t* sample_lens_host, int64_t B, int64_t S,
               const int32_t* targets_host, const int32_t* target_lens_host, int64_t U_max, int32_t* frame_labels_dev,
               float* frame_log_probs_dev, double* scores_dev, void* stream);

/* ---- transcribe: load -> mel -> model -> greedy (scripts/transcribe.py:69-82), batched.
 * tokens (B, L) int32, lens (B); L = vasr_num_tokens(vasr_num_frames(S)). */
int vasr_transcribe(vasr_handle* h, const float* pcm_dev, int64_t B, int64_t S,
                    int32_t* tokens_dev, int32_t* lens_dev, void* stream);
/* Host buffers in, host buffers out; H2D and D2H copies inside; synchronous. */
int vasr_transcribe_host(vasr_handle* h, const float* pcm_host, int64_t B, int64_t S,
                         int32_t* tokens_host, int32_t* lens_host);

/* ---- config 5: FakeQuantize of the 12 non-SSM modules (velocity_asr/quantize.py)
 * prepare_model_for_qat (quantize.py:269-322, ssm_state_fp32 = True) replaces temporal_binding.conv,
 * pool1/pool2.pool_proj, cross_attention.{q,k,v,out}_proj, fusion.{gate_proj.0,local_proj,global_proj,
 * out_proj} and ctc_head.proj.2 by QuantizedLinear / QuantizedConv1d: per-output-channel symmetric int8
 * FakeQuantize of the weight, fp32 matmul, per-tensor asymmetric uint8 FakeQuantize of the output
 * (quantize.py:180-191, 248-266).  vasr_set_quantization(h, 1) + vasr_commit_weights applies the weight side
 * (the module's own weights are kept, unlike the reference, which re-initialises them: SURVEY.md 5.8);
 * output nodes pass through until calibrated (quantize.py:82-84).
 * vasr_calibrate runs one forward on mel (B, T, mel_bins) with the output nodes in training mode: each takes
 * min / max of the tensor it is about to quantise, sets scale / zero point (quantize.py:99-121) and
 * quantises with them; the values stay for later forwards (calibrate_model, quantize.py:325-371).
 * module = reference module name, e.g. "ctc_head.proj.2". */
int vasr_set_quantization(vasr_handle* h, int enabled);
int vasr_calibrate(vasr_handle* h, const float* mel_dev, int64_t B, int64_t T, void* stream);
int vasr_get_quant_params(vasr_handle* h, const char* module, float* scale, float* zero_point);
int vasr_set_quant_params(vasr_handle* h, const char* module, float scale, float zero_point);
/* One quantised projection on its own (parity seam for QuantizedLinear.forward / QuantizedConv1d.forward,
 * quantize.py:180-191, 248-266): the projection that hosts `module` — fused neighbours included: k_proj | v_proj
 * share one, gate_proj.0 | local_proj | global_proj another (input [local | ctx]) — on x (B, R, K) with its
 * fake-quantised weights, bias and output FakeQuantize, no activation.  For temporal_binding.conv x is the mel
 * (B, R = T, mel_bins) and out has (R + 1) / 2 rows per utterance.  out: (B, R_out, N) with N the projection's
 * full width; *n_out, *col0, *ncol (may be NULL) receive N and the column range of `module` inside it. */
int vasr_quant_site(vasr_handle* h, const char* module, const float* x_dev, int64_t B, int64_t R, float* out_dev,
                    int32_t* n_out, int32_t* col0, int32_t* ncol, void* stream);

/* ---- a plain linear layer (F.linear), exposed so the GEMM kernel can be tested alone.
 * act: 0 none, 1 gelu(erf), 2 softplus, 3 sigmoid.  x (M, K) stride ldx, w (N, K), bias (N) or
 * NULL, out (M, N) stride ldo.  K % 16 == 0. */
int vasr_linear(const float* x_dev, int64_t ldx, const float* w_dev, const float* bias_dev,
                float* out_dev, int64_t ldo, int64_t M, int64_t K, int64_t N, int act, void* stream);

/* Same contract through the tensor-core kernel (tcgen05 + TMEM + TMA, 3xTF32 split): the
 * kernel every token-sized projection of the model runs on.  K % 4 == 0, N % 4 == 0.
 * The kernel reads the weight as two TF32 matrices [hi | lo] (2*N*K floats) made by
 * vasr_split_tf32; pass w_split_dev = NULL to have the call split w_dev on the fly. */
int vasr_split_tf32(const float* w_dev, float* split_dev, int64_t numel, void* stream);
/* resid_dev (M, N) with row stride ldr, or NULL: added after the activation (the residual adds of
 * ssm.py:418-425 are fused this way). */
int vasr_linear_tc(const float* x_dev, int64_t ldx, const float* w_dev, const float* w_split_dev,
                   const float* bias_dev, const float* resid_dev, int64_t ldr, float* out_dev, int64_t ldo,
                   int64_t M, int64_t K, int64_t N, int act, void* stream);

/* ---- bookkeeping for the bench: kernels launched by this handle since creation, and the
 * share of the last vasr_transcribe spent in the scan (device ms, CUDA events on `stream`)
 * when timing is enabled with vasr_set_timing(h, 1). */
int64_t vasr_kernel_launches(const vasr_handle* h);
int64_t vasr_tc_launches(const vasr_handle* h);   /* of which: tensor-core projection launches */
int vasr_set_timing(vasr_handle* h, int enabled);
int vasr_last_timing(const vasr_handle* h, float* scan_ms, int32_t* scan_launches, float* total_ms);
int64_t vasr_workspace_bytes(const vasr_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* VASR_H_ */
