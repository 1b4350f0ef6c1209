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
cudaError_t launch_beam_search_lm(const float* logits, const float2* stats, const LmView& lm, double lm_weight,
                                  int64_t B, int64_t L, int V, int W, int blank, int32_t* trie, float* trie_lm,
                                  int64_t trie_cap, float* rows, int32_t* out_tokens, int32_t* out_lens,
                                  double* out_scores, cudaStream_t s);

}  // namespace vasr
