// lm.cuh — device tables of an ARPA n-gram language model over token ids (lm.cu builds them, the seam kernel
// of lm.cu and the fused beam search of beam.cu read them).  Nothing outside these files sees the layout.
//
// Semantics (natural log, every stored value rounded once to fp32):
//   h = ("<s>",) + prefix, cut to its last order-1 items;
//   P(w | h) = p(h w) if listed, else bow(h) + P(w | h[1:]), bow(unlisted) = 0, unigram level: <unk> substitutes;
//   evaluated in fp64 from the listed entry that is found, adding the back-off weights from the shortest backed-off
//   context outward, then rounded to fp32.
// Layout: contexts are nodes of a trie over REVERSED histories (node 0 = the empty context; the child of node c
// by symbol s is the context with s prepended), so the listed suffixes of a history are found by walking from the
// root with its newest symbol first.  Tokens are 0 .. V-1, the context symbol <s> is V.  A context node has its
// fp32 back-off weight and a CSR list of its listed continuations (token ascending); the unigram level is a dense
// row with <unk> substituted.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

namespace vasr {

constexpr int kLmMaxOrder = 8;
constexpr unsigned long long kLmEmpty = ~0ull;

struct LmView {
  int order = 0, V = 0;
  int64_t hash_cap = 0;                        // power of two; key = (node << 32) | symbol -> child node
  const unsigned long long* hash_key = nullptr;
  const int32_t* hash_val = nullptr;
  const float* bow = nullptr;                  // (nodes)
  const int64_t* off = nullptr;                // (nodes + 1): continuations of node n are [off[n], off[n+1])
  const int32_t* cont_tok = nullptr;
  const float* cont_lp = nullptr;
  const float* uni = nullptr;                  // (V)
};

__host__ __device__ inline unsigned long long lm_hash(unsigned long long k) {   // splitmix64 finaliser
  k ^= k >> 30;
  k *= 0xbf58476d1ce4e5b9ull;
  k ^= k >> 27;
  k *= 0x94d049bb133111ebull;
  return k ^ (k >> 31);
}

__device__ __forceinline__ int lm_child(const LmView& lm, int node, int sym) {
  const unsigned long long key = ((unsigned long long)(unsigned)node << 32) | (unsigned)sym;
  unsigned long long h = lm_hash(key) & (unsigned long long)(lm.hash_cap - 1);
  for (;;) {
    const unsigned long long k = lm.hash_key[h];
    if (k == key) return lm.hash_val[h];
    if (k == kLmEmpty) return -1;
    h = (h + 1) & (unsigned long long)(lm.hash_cap - 1);
  }
}

// The listed suffixes of a history of k symbols (k <= order - 1); sym(i) is its i-th newest symbol (i >= 1),
// called in order and only while the suffixes are listed.  ctx[i] / bw[i] = node and back-off weight of the
// suffix of length i for i <= the returned m; bw[i] = 0 for m < i <= k (an unlisted context backs off for free).
template <class Sym>
__device__ __forceinline__ int lm_walk(const LmView& lm, int k, Sym sym, int (&ctx)[kLmMaxOrder],
                                       float (&bw)[kLmMaxOrder]) {
  int m = 0, c = 0;
#pragma unroll
  for (int i = 1; i < kLmMaxOrder; ++i) {
    ctx[i] = -1;
    bw[i] = 0.f;
    if (i <= k && m == i - 1) {
      const int c2 = lm_child(lm, c, sym(i));
      if (c2 >= 0) {
        c = c2;
        ctx[i] = c2;
        bw[i] = lm.bow[c2];
        m = i;
      }
    }
  }
  return m;
}

// fp32(base + bw[j+1] + ... + bw[k]) in fp64, shortest backed-off context first
__device__ __forceinline__ float lm_backoff(float base, int j, int k, const float (&bw)[kLmMaxOrder]) {
  double s = (double)base;
#pragma unroll
  for (int i = 1; i < kLmMaxOrder; ++i)
    if (i > j && i <= k) s = __dadd_rn(s, (double)bw[i]);
  return __double2float_rn(s);
}

// lm(history, tok) for a history of k symbols given as lm_walk takes it: the longest listed context that lists
// the token, then the back-off weights above it
template <class Sym>
__device__ __forceinline__ float lm_score(const LmView& lm, int k, Sym sym, int tok) {
  int ctx[kLmMaxOrder];
  float bw[kLmMaxOrder];
  const int m = lm_walk(lm, k, sym, ctx, bw);
  float base = lm.uni[tok];
  int j = 0;
#pragma unroll
  for (int q = kLmMaxOrder - 1; q >= 1; --q) {
    if (j == 0 && q <= m) {
      int64_t lo = lm.off[ctx[q]], hi = lm.off[ctx[q] + 1];
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (lm.cont_tok[mid] < tok) lo = mid + 1;
        else hi = mid;
      }
      if (lo < lm.off[ctx[q] + 1] && lm.cont_tok[lo] == tok) {
        base = lm.cont_lp[lo];
        j = q;
      }
    }
  }
  return lm_backoff(base, j, k, bw);
}

// ---- word LM over a character vocabulary ------------------------------------------------------------------
// The LM above with word ids as its symbols (word id = index in the file's unigram list, <s> = the context symbol
// V = word count), plus the spelling trie of its lexicon over token ids.  Node 0 is the empty spelling; a node has
// a CSR list of (token, child) pairs, token ascending, and the word it spells (or -1).
struct LexView {
  int delim = -1, constrained = 0;
  int unk = -1, eos = -1;                      // word ids of <unk> (-1: none) and of </s> (<unk>'s when unlisted)
  const int32_t* off = nullptr;                // (nodes + 1)
  const int32_t* tok = nullptr;                // (edges)
  const int32_t* child = nullptr;              // (edges)
  const int32_t* word = nullptr;               // (nodes)
};

// the child of spelling node `node` by token t, or -1 (also when node is -1: off the lexicon)
__device__ __forceinline__ int lex_child(const LexView& lx, int node, int t) {
  if (node < 0) return -1;
  int lo = lx.off[node], hi = lx.off[node + 1];
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (lx.tok[mid] < t) lo = mid + 1;
    else hi = mid;
  }
  return lo < lx.off[node + 1] && lx.tok[lo] == t ? lx.child[lo] : -1;
}

// ---- host side (lm.cu) ------------------------------------------------------------------------------------
struct LmHostTables {
  int order = 0, V = 0;
  int64_t listed = 0, kept = 0;                // n-gram lines in the file / reachable ones kept
  std::vector<unsigned long long> hash_key;
  std::vector<int32_t> hash_val;
  std::vector<float> bow, cont_lp, uni;
  std::vector<int64_t> off;
  std::vector<int32_t> cont_tok;
};
// Parses an ARPA file; no device call.  Returns false with a message naming the line on malformed input.
bool lm_parse_arpa(const char* path, const char* const* vocab, int V, int blank, LmHostTables* t, std::string* err);
// One device allocation holding every table of `t`; *view points into it.
cudaError_t lm_upload(const LmHostTables& t, void** block, LmView* view);
// out[i] = lm(prefix_i, tokens[i]); prefixes (n, max(order-1, 1)) int32 holds the last min(len, order-1) tokens
// of prefix i right-aligned (its newest token last), lens[i] its true length.  Tokens outside [0, V) give NaN.
cudaError_t launch_lm_log_prob(const LmView& lm, const int32_t* prefixes, const int32_t* lens, int64_t n,
                               const int32_t* tokens, float* out, cudaStream_t s);
// The prefix beam search with the LM fused (beam.cu); stats from launch_beam_rows.  trie: 5 x (B, trie_cap) int32
// (parent | token | depth | first child | next sibling), trie_lm (B, trie_cap) fp32, rows (B, W, V) fp32 scratch.
// lens / lens_stride: the optional per-utterance frame counts of launch_beam_search.
cudaError_t launch_beam_search_lm(const float* logits, const float2* stats, const LmView& lm, double lm_weight,
                                  int64_t B, int64_t L, const int32_t* lens, int lens_stride, int V, int W, int blank,
                                  int32_t* trie, float* trie_lm, int64_t trie_cap, float* rows, int32_t* out_tokens,
                                  int32_t* out_lens, double* out_scores, cudaStream_t s);

struct LexHostTables {
  std::vector<std::string> words;              // word id -> string (the unigram words, <s> excluded, file order)
  int64_t lexicon = 0;                         // spellable words other than <s>, </s>, <unk>
  int delim = -1, unk = -1, eos = -1;
  std::vector<int32_t> off, tok, child, word;
};
// Parses a word-level ARPA file (lm_parse_arpa over the file's own unigram words) and builds the spelling trie of
// its lexicon over `vocab`; no device call.  Returns false with a message on a bad delimiter, a malformed file
// (naming the line), a lexicon-free model without <unk> or a constrained one with an empty lexicon.
bool lm_parse_word_arpa(const char* path, const char* const* vocab, int V, int blank, const char* delimiter,
                        bool constrained, LmHostTables* t, LexHostTables* x, std::string* err);
cudaError_t lex_upload(const LexHostTables& x, bool constrained, void** block, LexView* view);
// The prefix beam search with a word LM fused (beam.cu).  top_tok (B*L, K) from launch_beam_rows (lexicon-free mode
// only, K = min(W + 2, V - 1)); trie: 9 x (B, trie_cap) int32, trie_f (B, trie_cap) fp32.
// lens / lens_stride as in launch_beam_search; the end-of-utterance step follows each utterance's last frame.
cudaError_t launch_beam_search_word_lm(const float* logits, const float2* stats, const int32_t* top_tok, int K,
                                       const LmView& lm, const LexView& lx, double lm_weight, double word_score,
                                       int64_t B, int64_t L, const int32_t* lens, int lens_stride, int V, int W,
                                       int blank, int32_t* trie, float* trie_f, int64_t trie_cap, int32_t* out_tokens,
                                       int32_t* out_lens, double* out_scores, cudaStream_t s);

}  // namespace vasr
