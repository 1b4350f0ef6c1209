// beam.cu — CTC prefix beam search on the device (ctc_beam_search, velocity_asr/decode.py:128-217, the
// lm_scorer=None path).  The reference walks every (beam, token) pair of every frame in Python; its rule is
//   new_beams[key] = max over candidates of (score + log_prob), first-inserted wins a tie,
//   key = prefix (blank, or the beam's own last token again) | prefix + (token,)
//   then the `beam_width` best keys, stable in insertion order.
// Two facts make that cheap without changing a single result:
//  * inside one beam the extension candidates are ranked by the frame's log-probs alone, so a candidate that
//    makes the global top-W is among the frame's W+1 best non-blank tokens (one of them may be the beam's
//    last token, which does not extend).  beam_rows_kernel finds those per frame, all frames in parallel;
//  * two candidates share a key only when an extension recreates a prefix that is already a beam (the child
//    of the extending beam) — found through a per-utterance trie of prefixes (parent, token, depth).
// beam_search_kernel then runs the frames in order, one warp per utterance, one beam per lane, scores in
// fp64 (the reference adds Python floats), ties broken by the reference's insertion order
// (beam rank, then blank, then token id).
//
// With an n-gram LM (beam_search_lm_kernel), an offer that extends a prefix scores
//   (score + lp[tok]) + lm_weight * lm(prefix, tok)          fp64, in this order;
// blank and repeat offers are unchanged.  One CTA per utterance, one warp per beam:
//  * each beam keeps a dense fp32 row lm(prefix, .) over V in a slot of global memory.  A row is built only when
//    a new prefix is created (at most W per frame) from the LM's suffix chain and continuation lists; blank and
//    repeat survivors keep their prefix, their slot and their row;
//  * each beam's warp lists its own W+1 best extension tokens by the fused offer (ties -> lower token id).  W+1
//    still suffices: every entry ranked above a token x in that list is the beam's last token, or a token whose
//    child prefix is already a beam — and that child's key scores at least the parent's offer (max-merge) and
//    was inserted no later, so it outranks x too — or another extension that outranks x.  So if x makes the
//    global top-W, at most W-1 entries above it are extensions or child keys, plus possibly `last`, whose repeat
//    offer carries no LM term and need not dominate x: x is among the first W+1;
//  * the parent's offer to a child beam needs lm(parent prefix, token), a property of the child's prefix: it is
//    stored in the trie node when the node is created;
//  * the rank / merge / selection loop is beam_search_kernel's, run by warp 0 (one lane per beam), with one change:
//    trie nodes are canonical.  An extension that recreates a prefix seen before (it dropped out of the beams and
//    comes back) reuses that prefix's node, found in its parent's child list, so "beam j's parent node is beam i's
//    node" means "beam j's prefix extends beam i's" even then.  With an LM prefixes drop out and return often, and
//    a fresh node would hide a surviving child from its recreated parent (two offers to one prefix, unmerged).
#include <float.h>

#include "common.cuh"
#include "kernels.cuh"
#include "lm.cuh"

namespace vasr {

namespace {

// Ragged batches: every kernel below takes an optional per-utterance frame count, read as (pointer, stride) so
// the ragged dims of a fused call (kernels.cuh, RAG_L) serve without a copy.  Utterance b is then searched over
// its rows b * L + [0, len_b) only; the row stride stays L.  A null pointer means len_b = L for every utterance.
__device__ __forceinline__ int64_t utt_frames(const int32_t* lens, int stride, int64_t b, int64_t L) {
  return lens ? (int64_t)lens[b * stride] : L;
}

// One warp per (utterance, frame) row: max, log-sum-exp, and the K best non-blank tokens by
// log-prob (ties -> lower token id).  log-prob = (x - max) - log(sum exp(x - max)), torch's order.
// Rows at or past their utterance's length are neither read nor written.
__global__ void __launch_bounds__(256) beam_rows_kernel(const float* __restrict__ logits, float2* __restrict__ stats,
                                                        int32_t* __restrict__ top_tok, int64_t M, int V, int K,
                                                        int blank, int64_t L, const int32_t* __restrict__ lens,
                                                        int lens_stride) {
  const int lane = threadIdx.x & 31;
  const int64_t m = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (m >= M) return;
  if (lens && m % L >= utt_frames(lens, lens_stride, m / L, L)) return;
  const float* x = logits + m * V;
  float mx = -INFINITY;
  for (int n = lane; n < V; n += 32) mx = fmaxf(mx, x[n]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
  for (int n = lane; n < V; n += 32) sum += expf(x[n] - mx);
  sum = warp_sum(sum);
  const float ls = logf(sum);
  if (lane == 0) stats[m] = make_float2(mx, ls);
  // K passes; pass k takes the best entry strictly after the previous winner in (lp desc, token asc) order
  float pv = INFINITY;
  int pi = -1;
  for (int k = 0; k < K; ++k) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int n = lane; n < V; n += 32) {
      if (n == blank) continue;
      const float v = (x[n] - mx) - ls;
      const bool after = v < pv || (v == pv && n > pi);
      if (after && (bi == 0x7fffffff || v > bv)) {  // ascending n inside a lane: first seen wins ties
        bv = v;
        bi = n;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi != 0x7fffffff && (bi == 0x7fffffff || ov > bv || (ov == bv && oi < bi))) {
        bv = ov;
        bi = oi;
      }
    }
    if (lane == 0) top_tok[m * K + k] = bi == 0x7fffffff ? -1 : bi;
    if (bi == 0x7fffffff) {
      for (int kk = k + 1; kk < K; ++kk)
        if (lane == 0) top_tok[m * K + kk] = -1;
      break;
    }
    pv = bv;
    pi = bi;
  }
}

constexpr long long kNoOrder = 0x7fffffffffffffffLL;

__global__ void __launch_bounds__(32) beam_search_kernel(
    const float* __restrict__ logits, const float2* __restrict__ stats, const int32_t* __restrict__ top_tok, int K,
    int64_t L, const int32_t* __restrict__ lens, int lens_stride, int V, int W, int blank, int32_t* trie_parent,
    int32_t* trie_token, int32_t* trie_depth, int64_t trie_cap, int32_t* __restrict__ out_tokens,
    int32_t* __restrict__ out_lens, double* __restrict__ out_scores) {
  const int64_t b = blockIdx.x;
  const int lane = threadIdx.x;
  const int64_t Lb = utt_frames(lens, lens_stride, b, L);
  int32_t* parent = trie_parent + b * trie_cap;
  int32_t* token = trie_token + b * trie_cap;
  int32_t* depth = trie_depth + b * trie_cap;

  __shared__ int s_node[32], s_last[32], s_pl[32], s_tk[32], n_node[32], n_last[32];
  __shared__ double s_score[32], n_score[32];

  if (lane == 0) {
    parent[0] = -1;
    token[0] = -1;
    depth[0] = 0;
  }
  int nb = 1, n_nodes = 1;
  int node = 0, last = -1;  // last = -1 is the reference's None
  double score = 0.0;
  const long long Vp = (long long)V + 1;
  __syncwarp();

  for (int64_t t = 0; t < Lb; ++t) {
    const int64_t row = b * L + t;
    const float* x = logits + row * V;
    const float2 st = stats[row];
    const int32_t* tt = top_tok + row * K;
    auto lp = [&](int tok) -> double { return (double)((x[tok] - st.x) - st.y); };
    const bool valid = lane < nb;

    s_node[lane] = valid ? node : -2;
    const int par = valid ? parent[node] : -3;
    const int tk = valid ? token[node] : -1;
    __syncwarp();
    int pl = -1;
    if (valid && par >= 0)
      for (int j = 0; j < nb; ++j)
        if (s_node[j] == par) pl = j;
    s_pl[lane] = pl;
    s_tk[lane] = tk;
    s_last[lane] = last;
    s_score[lane] = score;
    __syncwarp();

    // the key this beam already owns: its own blank / repeat candidates and, when its parent prefix is a
    // beam too, the parent's extension by this beam's last prefix token
    double e_score = -INFINITY;
    int e_last = blank;
    long long e_order = kNoOrder;
    bool e_avail = valid;
    if (valid) {
      double cs[3];
      int cl[3];
      long long co[3];
      bool ch[3];
      const bool h1 = pl >= 0 && s_last[pl] != tk;
      const double sc1 = h1 ? s_score[pl] + lp(tk) : 0.0;
      const long long o1 = (long long)pl * Vp + 1 + tk;
      const bool h3 = last >= 0 && last != blank;
      const double sc3 = h3 ? score + lp(last) : 0.0;
      const int first = (h1 && pl < lane) ? 0 : 2;  // where the parent's candidate sits in insertion order
      const int i2 = first == 0 ? 1 : 0, i3 = i2 + 1;
      cs[first] = sc1, cl[first] = tk, co[first] = o1, ch[first] = h1;
      cs[i2] = score + lp(blank), cl[i2] = blank, co[i2] = (long long)lane * Vp, ch[i2] = true;
      cs[i3] = sc3, cl[i3] = last, co[i3] = (long long)lane * Vp + 1 + last, ch[i3] = h3;
      bool none = true;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        if (!ch[i]) continue;
        if (none || cs[i] > e_score) {
          e_score = cs[i];
          e_last = cl[i];
        }
        if (none) e_order = co[i];
        none = false;
      }
    }

    // this beam's extensions to prefixes that are not beams yet, best first
    int p = valid ? 0 : K;
    int x_tok = -1;
    double x_score = -INFINITY;
    auto advance = [&]() {
      while (p < K) {
        const int tok = tt[p];
        if (tok < 0) {
          p = K;
          break;
        }
        bool skip = tok == last;
        for (int j = 0; j < nb && !skip; ++j) skip = s_pl[j] == lane && s_tk[j] == tok;
        if (!skip) {
          x_tok = tok;
          x_score = score + lp(tok);
          return;
        }
        ++p;
      }
    };
    advance();

    int count = 0;
    for (int r = 0; r < W; ++r) {
      const bool hx = p < K;
      const long long x_order = (long long)lane * Vp + 1 + x_tok;
      bool take_e = e_avail;
      if (e_avail && hx) take_e = e_score > x_score || (e_score == x_score && e_order < x_order);
      double ps = take_e ? e_score : (hx ? x_score : -INFINITY);
      long long po = take_e ? e_order : (hx ? x_order : kNoOrder);
      double bs = ps;
      long long bo = po;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double os = __shfl_xor_sync(0xffffffffu, bs, o);
        const long long oo = __shfl_xor_sync(0xffffffffu, bo, o);
        if (oo != kNoOrder && (bo == kNoOrder || os > bs || (os == bs && oo < bo))) {
          bs = os;
          bo = oo;
        }
      }
      if (bo == kNoOrder) break;
      const bool mine = po == bo;
      const bool is_new = mine && !take_e;
      const unsigned newm = __ballot_sync(0xffffffffu, is_new);
      if (mine) {
        if (take_e) {
          n_node[r] = node;
          n_score[r] = e_score;
          n_last[r] = e_last;
          e_avail = false;
        } else {
          parent[n_nodes] = node;
          token[n_nodes] = x_tok;
          depth[n_nodes] = depth[node] + 1;
          n_node[r] = n_nodes;
          n_score[r] = x_score;
          n_last[r] = x_tok;
          ++p;
          advance();
        }
      }
      n_nodes += newm != 0;
      ++count;
    }
    __syncwarp();
    nb = count;
    if (lane < nb) {
      node = n_node[lane];
      score = n_score[lane];
      last = n_last[lane];
    }
    __syncwarp();
  }

  if (lane < W) {
    int32_t* out = out_tokens + (b * W + lane) * L;
    if (lane < nb) {
      const int len = depth[node];
      out_scores[b * W + lane] = score;
      out_lens[b * W + lane] = len;
      int nd = node;
      for (int i = len - 1; i >= 0; --i) {
        out[i] = token[nd];
        nd = parent[nd];
      }
      for (int64_t i = len; i < L; ++i) out[i] = -1;
    } else {
      out_scores[b * W + lane] = -INFINITY;
      out_lens[b * W + lane] = -1;
      for (int64_t i = 0; i < L; ++i) out[i] = -1;
    }
  }
}

// ---- the search with an n-gram LM ----------------------------------------------------------------------------
constexpr int kLaneTop = 4;   // entries each lane buffers while a warp lists a beam's candidates

// row[tok] = lm(prefix of `node`, tok) for every tok: the unigram row backed off through the whole history, then
// the continuation lists of the listed suffixes, shortest first, so a longer listed context overwrites
__device__ __forceinline__ void lm_build_row(const LmView& lm, const int32_t* parent, const int32_t* token,
                                             const int32_t* depth, int node, float* row, int lane) {
  const int d = depth[node];
  const int k = min(lm.order - 1, d + 1);
  int nd = node;
  int ctx[kLmMaxOrder];
  float bw[kLmMaxOrder];
  const int m = lm_walk(lm, k, [&](int q) {
    if (q > d) return lm.V;   // <s>
    const int s = token[nd];
    nd = parent[nd];
    return s;
  }, ctx, bw);
  for (int tok = lane; tok < lm.V; tok += 32) row[tok] = lm_backoff(lm.uni[tok], 0, k, bw);
  __syncwarp();
#pragma unroll
  for (int j = 1; j < kLmMaxOrder; ++j) {
    if (j <= m) {
      const int64_t e1 = lm.off[ctx[j] + 1];
      for (int64_t e = lm.off[ctx[j]] + lane; e < e1; e += 32) row[lm.cont_tok[e]] = lm_backoff(lm.cont_lp[e], j, k, bw);
    }
    __syncwarp();
  }
}

// One beam's K best extension tokens by fused offer (ties -> lower token id) -> c_tok / c_sc / c_lm[0 .. K), -1
// padded.  Each lane buffers the kLaneTop best of its own tokens and refills after its last taken entry when the
// buffer runs dry; the warp takes the best buffered head K times.
__device__ __forceinline__ void lm_candidates(const float* x, float2 st, const float* row, double score, double lmw,
                                              int V, int K, int blank, int lane, int* c_tok, double* c_sc,
                                              float* c_lm) {
  auto offer = [&](int tok) {
    const double lp = (double)((x[tok] - st.x) - st.y);
    return __dadd_rn(__dadd_rn(score, lp), __dmul_rn(lmw, (double)row[tok]));
  };
  double hv[kLaneTop];
  int hi[kLaneTop];
  double pv = INFINITY;
  int pi = -1;
  bool more = false;
  auto refill = [&]() {
#pragma unroll
    for (int q = 0; q < kLaneTop; ++q) {
      hv[q] = -INFINITY;
      hi[q] = -1;
    }
    int cnt = 0;
    for (int tok = lane; tok < V; tok += 32) {
      if (tok == blank) continue;
      const double v = offer(tok);
      if (pi >= 0 && !(v < pv || (v == pv && tok > pi))) continue;   // taken already
      ++cnt;
      if (hi[kLaneTop - 1] >= 0 && !(v > hv[kLaneTop - 1])) continue;   // tokens ascend: a tie goes after
      hv[kLaneTop - 1] = v;
      hi[kLaneTop - 1] = tok;
#pragma unroll
      for (int q = kLaneTop - 1; q > 0; --q) {
        if (hi[q - 1] < 0 || hv[q] > hv[q - 1]) {
          const double tv = hv[q];
          hv[q] = hv[q - 1];
          hv[q - 1] = tv;
          const int ti = hi[q];
          hi[q] = hi[q - 1];
          hi[q - 1] = ti;
        }
      }
    }
    more = cnt > kLaneTop;
  };
  refill();
  for (int k = 0; k < K; ++k) {
    double bv = hv[0];
    int bi = hi[0];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (bi < 0 || ov > bv || (ov == bv && oi < bi))) {
        bv = ov;
        bi = oi;
      }
    }
    if (bi < 0) {
      for (int kk = k + lane; kk < K; kk += 32) c_tok[kk] = -1;
      break;
    }
    if (hi[0] == bi) {   // the lane that owns the token
      c_tok[k] = bi;
      c_sc[k] = bv;
      c_lm[k] = row[bi];
      pv = bv;
      pi = bi;
#pragma unroll
      for (int q = 0; q < kLaneTop - 1; ++q) {
        hv[q] = hv[q + 1];
        hi[q] = hi[q + 1];
      }
      hv[kLaneTop - 1] = -INFINITY;
      hi[kLaneTop - 1] = -1;
      if (hi[0] < 0 && more) refill();
    }
  }
}

__global__ void __launch_bounds__(512) beam_search_lm_kernel(
    const float* __restrict__ logits, const float2* __restrict__ stats, const LmView lm, double lmw, int K,
    int64_t L, const int32_t* __restrict__ lens, int lens_stride, int V, int W, int blank, int32_t* trie_parent,
    int32_t* trie_token, int32_t* trie_depth, int32_t* trie_child, int32_t* trie_sibling, float* trie_lm,
    int64_t trie_cap, float* rows, int32_t* __restrict__ out_tokens, int32_t* __restrict__ out_lens,
    double* __restrict__ out_scores) {
  const int64_t b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const int64_t Lb = utt_frames(lens, lens_stride, b, L);
  int32_t* parent = trie_parent + b * trie_cap;
  int32_t* token = trie_token + b * trie_cap;
  int32_t* depth = trie_depth + b * trie_cap;
  int32_t* first_child = trie_child + b * trie_cap;
  int32_t* next_sibling = trie_sibling + b * trie_cap;
  float* node_lm = trie_lm + b * trie_cap;   // lm(parent prefix, token) of each node
  float* urows = rows + b * (int64_t)W * V;

  // warp 0's selection state, as in beam_search_kernel
  __shared__ int s_node[32], s_last[32], s_pl[32], s_tk[32], n_node[32], n_last[32], n_slot[32];
  __shared__ double s_score[32], n_score[32];
  // each beam's candidate list
  __shared__ int c_tok[32][33];
  __shared__ double c_sc[32][33];
  __shared__ float c_lm[32][33];
  // the beams as every warp sees them
  __shared__ int b_node[32], b_slot[32], b_new[32], b_nb;
  __shared__ double b_score[32];

  if (threadIdx.x == 0) {
    parent[0] = -1;
    token[0] = -1;
    depth[0] = 0;
    first_child[0] = -1;
    node_lm[0] = 0.f;
    b_node[0] = 0;
    b_slot[0] = 0;
    b_new[0] = 1;
    b_score[0] = 0.0;
    b_nb = 1;
  }
  int nb = 1, n_nodes = 1;
  int node = 0, last = -1, slot = 0;
  double score = 0.0;
  const long long Vp = (long long)V + 1;
  __syncthreads();

  for (int64_t t = 0; t < Lb; ++t) {
    const int64_t rw = b * L + t;
    const float* x = logits + rw * V;
    const float2 st = stats[rw];
    for (int w = warp; w < b_nb; w += nwarps) {
      float* row = urows + (int64_t)b_slot[w] * V;
      if (b_new[w]) lm_build_row(lm, parent, token, depth, b_node[w], row, lane);
      lm_candidates(x, st, row, b_score[w], lmw, V, K, blank, lane, c_tok[w], c_sc[w], c_lm[w]);
    }
    __syncthreads();

    if (warp == 0) {
      auto lp = [&](int tok) -> double { return (double)((x[tok] - st.x) - st.y); };
      const bool valid = lane < nb;

      s_node[lane] = valid ? node : -2;
      const int par = valid ? parent[node] : -3;
      const int tk = valid ? token[node] : -1;
      __syncwarp();
      int pl = -1;
      if (valid && par >= 0)
        for (int j = 0; j < nb; ++j)
          if (s_node[j] == par) pl = j;
      s_pl[lane] = pl;
      s_tk[lane] = tk;
      s_last[lane] = last;
      s_score[lane] = score;
      __syncwarp();

      double e_score = -INFINITY;
      int e_last = blank;
      long long e_order = kNoOrder;
      bool e_avail = valid;
      if (valid) {
        double cs[3];
        int cl[3];
        long long co[3];
        bool ch[3];
        const bool h1 = pl >= 0 && s_last[pl] != tk;
        const double sc1 = h1 ? __dadd_rn(__dadd_rn(s_score[pl], lp(tk)), __dmul_rn(lmw, (double)node_lm[node])) : 0.0;
        const long long o1 = (long long)pl * Vp + 1 + tk;
        const bool h3 = last >= 0 && last != blank;
        const double sc3 = h3 ? score + lp(last) : 0.0;
        const int first = (h1 && pl < lane) ? 0 : 2;
        const int i2 = first == 0 ? 1 : 0, i3 = i2 + 1;
        cs[first] = sc1, cl[first] = tk, co[first] = o1, ch[first] = h1;
        cs[i2] = score + lp(blank), cl[i2] = blank, co[i2] = (long long)lane * Vp, ch[i2] = true;
        cs[i3] = sc3, cl[i3] = last, co[i3] = (long long)lane * Vp + 1 + last, ch[i3] = h3;
        bool none = true;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          if (!ch[i]) continue;
          if (none || cs[i] > e_score) {
            e_score = cs[i];
            e_last = cl[i];
          }
          if (none) e_order = co[i];
          none = false;
        }
      }

      int p = valid ? 0 : K;
      int x_tok = -1;
      double x_score = -INFINITY;
      auto advance = [&]() {
        while (p < K) {
          const int tok = c_tok[lane][p];
          if (tok < 0) {
            p = K;
            break;
          }
          bool skip = tok == last;
          for (int j = 0; j < nb && !skip; ++j) skip = s_pl[j] == lane && s_tk[j] == tok;
          if (!skip) {
            x_tok = tok;
            x_score = c_sc[lane][p];
            return;
          }
          ++p;
        }
      };
      advance();

      int count = 0;
      for (int r = 0; r < W; ++r) {
        const bool hx = p < K;
        const long long x_order = (long long)lane * Vp + 1 + x_tok;
        bool take_e = e_avail;
        if (e_avail && hx) take_e = e_score > x_score || (e_score == x_score && e_order < x_order);
        double ps = take_e ? e_score : (hx ? x_score : -INFINITY);
        long long po = take_e ? e_order : (hx ? x_order : kNoOrder);
        double bs = ps;
        long long bo = po;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const double os = __shfl_xor_sync(0xffffffffu, bs, o);
          const long long oo = __shfl_xor_sync(0xffffffffu, bo, o);
          if (oo != kNoOrder && (bo == kNoOrder || os > bs || (os == bs && oo < bo))) {
            bs = os;
            bo = oo;
          }
        }
        if (bo == kNoOrder) break;
        const bool mine = po == bo;
        bool created = false;
        if (mine) {
          if (take_e) {
            n_node[r] = node;
            n_score[r] = e_score;
            n_last[r] = e_last;
            n_slot[r] = slot;
            e_avail = false;
          } else {
            int c = first_child[node];
            while (c >= 0 && token[c] != x_tok) c = next_sibling[c];
            if (c < 0) {
              c = n_nodes;
              parent[c] = node;
              token[c] = x_tok;
              depth[c] = depth[node] + 1;
              node_lm[c] = c_lm[lane][p];
              first_child[c] = -1;
              next_sibling[c] = first_child[node];
              first_child[node] = c;
              created = true;
            }
            n_node[r] = c;
            n_score[r] = x_score;
            n_last[r] = x_tok;
            n_slot[r] = -1;
            ++p;
            advance();
          }
        }
        n_nodes += __ballot_sync(0xffffffffu, created) != 0;
        ++count;
      }
      __syncwarp();
      nb = count;
      int ns = -1;
      if (lane < nb) {
        node = n_node[lane];
        score = n_score[lane];
        last = n_last[lane];
        ns = n_slot[lane];
      }
      // survivors keep their row slot; new prefixes take the free ones, in beam order
      const bool fresh = lane < nb && ns < 0;
      const unsigned used = __reduce_or_sync(0xffffffffu, (lane < nb && ns >= 0) ? 1u << ns : 0u);
      const unsigned freshm = __ballot_sync(0xffffffffu, fresh);
      if (fresh) {
        unsigned fr = ~used;
        for (int q = __popc(freshm & ((1u << lane) - 1u)); q > 0; --q) fr &= fr - 1u;
        ns = __ffs(fr) - 1;
      }
      slot = ns;
      if (lane < nb) {
        b_node[lane] = node;
        b_slot[lane] = slot;
        b_new[lane] = fresh;
        b_score[lane] = score;
      }
      if (lane == 0) b_nb = nb;
    }
    __syncthreads();
  }

  if (warp == 0 && lane < W) {
    int32_t* out = out_tokens + (b * W + lane) * L;
    if (lane < nb) {
      const int len = depth[node];
      out_scores[b * W + lane] = score;
      out_lens[b * W + lane] = len;
      int nd = node;
      for (int i = len - 1; i >= 0; --i) {
        out[i] = token[nd];
        nd = parent[nd];
      }
      for (int64_t i = len; i < L; ++i) out[i] = -1;
    } else {
      out_scores[b * W + lane] = -INFINITY;
      out_lens[b * W + lane] = -1;
      for (int64_t i = 0; i < L; ++i) out[i] = -1;
    }
  }
}

// ---- the search with a word LM ---------------------------------------------------------------------------------
// Words are spelled in the character vocabulary and closed by the delimiter d (include/vasr.h states the rule).
// Only the offer by d that closes a non-empty pending run u carries a term, ((score + lp[d]) + lm_weight *
// lm(h, word(u))) + word_score; every other extension scores score + lp[tok].  In constrained mode a beam may only
// offer tokens that keep u on a lexicon word's spelling, and d only when u is empty or a lexicon word.
// One CTA per utterance, one warp per beam, beam_search_lm_kernel's canonical trie and warp 0's rank / merge /
// selection loop, but no V-wide LM rows.  Each trie node holds, set when it is created: its spelling-trie node
// (0: u is empty, -1: u is off the lexicon), the latest node at or above it whose token closed a word, the word
// that token closed, and how many words its prefix has closed — so the word history is a walk up closing nodes.
// lm(h, word(u)) is cached per node the first time a beam sits on it.
// W+1 suffices again: among a beam's offers the non-d ones rank by lp alone (the same score is added), and d is
// a single extra entry.  In lexicon-free mode every non-blank token is allowed, so a non-d token outside the
// frame's W+2 best non-blank tokens (beam_rows_kernel, ties -> lower id) has at least W+1 non-d offers above it
// in the beam's list; in constrained mode the allowed non-d tokens are the spelling node's children.  So the
// beam's W+1 best fused offers are among those tokens plus d, and the argument of beam_search_lm_kernel (every
// entry above a token x is `last`, a child key that outranks x, or an extension that outranks x) shows that a
// token making the global top W is among the beam's first W+1.  The parent's offer to a child beam is the same
// function of the parent's state.  After the last frame: close each beam's pending run (constrained: drop the
// beam when it is not a lexicon word), add lm_weight * lm(h, </s>), and sort the beams stably by that score.
struct WordTrie {
  int32_t *parent, *token, *depth, *first_child, *next_sibling;
  int32_t *lex, *closer, *word, *nwords;   // spelling node, latest closing node (-1: none), word closed, words so far
  float* close_lm;                         // lm(h, word(u)) of the node's prefix, NaN until computed
};

// lm(h(node) [+ extra], w): the node's word history, with `extra` (>= 0) appended as the newest word
__device__ __forceinline__ float word_lm(const LmView& lm, const WordTrie& tr, int node, int extra, int w) {
  int hn = tr.closer[node];
  bool first = extra >= 0;
  const int k = min(lm.order - 1, tr.nwords[node] + (first ? 1 : 0) + 1);
  return lm_score(lm, k, [&](int) {
    if (first) {
      first = false;
      return extra;
    }
    if (hn < 0) return lm.V;   // <s>
    const int s = tr.word[hn];
    hn = tr.closer[tr.parent[hn]];
    return s;
  }, w);
}

__device__ __forceinline__ int word_of(const LexView& lx, int ln) {
  const int w = ln >= 0 ? lx.word[ln] : -1;
  return w >= 0 ? w : lx.unk;
}

// the offer by d from a beam: ((score + lp) + lmw * lm) + ws when it closes a word, else score + lp
__device__ __forceinline__ double word_offer(double score, double lp, bool closes, float lm, double lmw, double ws) {
  const double s = __dadd_rn(score, lp);
  return closes ? __dadd_rn(__dadd_rn(s, __dmul_rn(lmw, (double)lm)), ws) : s;
}

__global__ void __launch_bounds__(512, 1) beam_search_word_lm_kernel(
    const float* __restrict__ logits, const float2* __restrict__ stats, const int32_t* __restrict__ top_tok, int K,
    const LmView lm, const LexView lx, double lmw, double ws, int64_t L, const int32_t* __restrict__ lens,
    int lens_stride, int V, int W, int blank, int32_t* trie, float* trie_f, int64_t trie_cap,
    int32_t* __restrict__ out_tokens, int32_t* __restrict__ out_lens, double* __restrict__ out_scores) {
  const int64_t b = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  const int64_t Lb = utt_frames(lens, lens_stride, b, L);   // the end-of-utterance step follows frame Lb - 1
  const int64_t pb = (int64_t)gridDim.x * trie_cap;   // one plane of the trie
  int32_t* base = trie + b * trie_cap;
  const WordTrie tr{base,          base + pb,     base + 2 * pb, base + 3 * pb, base + 4 * pb,
                    base + 5 * pb, base + 6 * pb, base + 7 * pb, base + 8 * pb, trie_f + b * trie_cap};
  const int d = lx.delim;
  const int KC = W + 1;   // entries of each beam's candidate list

  __shared__ int s_node[32], s_last[32], s_pl[32], s_tk[32], n_node[32], n_last[32];
  __shared__ double s_score[32], n_score[32];
  __shared__ int c_tok[32][33], c_lex[32][33];
  __shared__ double c_sc[32][33];
  __shared__ int b_node[32], b_lex[32], b_nb;
  __shared__ float b_dlm[32];
  __shared__ double b_score[32];

  if (threadIdx.x == 0) {
    tr.parent[0] = -1;
    tr.token[0] = -1;
    tr.depth[0] = 0;
    tr.first_child[0] = -1;
    tr.lex[0] = 0;
    tr.closer[0] = -1;
    tr.nwords[0] = 0;
    tr.close_lm[0] = __int_as_float(0x7fffffff);
    b_node[0] = 0;
    b_score[0] = 0.0;
    b_nb = 1;
  }
  int nb = 1, n_nodes = 1;
  int node = 0, last = -1;
  double score = 0.0;
  const long long Vp = (long long)V + 1;
  __syncthreads();

  for (int64_t t = 0; t < Lb; ++t) {
    const int64_t rw = b * L + t;
    const float* x = logits + rw * V;
    const float2 st = stats[rw];
    auto lp = [&](int tok) -> double { return (double)((x[tok] - st.x) - st.y); };

    // each beam's W+1 best offers, selection passes over its allowed tokens plus d (ties -> lower token id)
    for (int w = warp; w < b_nb; w += nwarps) {
      const int bn = b_node[w];
      const double s = b_score[w];
      const int ln = tr.lex[bn];
      const bool d_ok = ln == 0 || !lx.constrained || (ln > 0 && lx.word[ln] >= 0);
      const bool closes = ln != 0;
      float dlm = 0.f;
      if (closes && d_ok) {
        dlm = tr.close_lm[bn];
        if (isnan(dlm)) {
          if (lane == 0) {
            dlm = word_lm(lm, tr, bn, -1, word_of(lx, ln));
            tr.close_lm[bn] = dlm;
          }
          dlm = __shfl_sync(0xffffffffu, dlm, 0);
        }
      }
      const int lo = lx.constrained ? lx.off[ln] : 0;
      const int n = (lx.constrained ? lx.off[ln + 1] - lo : K) + 1;   // the last entry is d
      const int32_t* top = top_tok + rw * K;
      auto cand = [&](int i, int& tok, double& v) {
        if (i == n - 1) {
          tok = d;
          v = word_offer(s, lp(d), closes, dlm, lmw, ws);
          return d_ok;
        }
        tok = lx.constrained ? lx.tok[lo + i] : top[i];
        v = __dadd_rn(s, tok >= 0 ? lp(tok) : 0.0);
        return tok >= 0 && tok != d;
      };
      double pv = INFINITY;
      int pi = -1, cnt = 0;
      for (int k = 0; k < KC; ++k) {
        double bv = -INFINITY;
        int bi = 0x7fffffff;
        for (int i = lane; i < n; i += 32) {
          int tok;
          double v;
          if (!cand(i, tok, v)) continue;
          const bool after = v < pv || (v == pv && tok > pi);
          if (after && (bi == 0x7fffffff || v > bv || (v == bv && tok < bi))) {
            bv = v;
            bi = tok;
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const double ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (oi != 0x7fffffff && (bi == 0x7fffffff || ov > bv || (ov == bv && oi < bi))) {
            bv = ov;
            bi = oi;
          }
        }
        if (bi == 0x7fffffff) break;
        if (lane == 0) {
          c_tok[w][k] = bi;
          c_sc[w][k] = bv;
        }
        pv = bv;
        pi = bi;
        ++cnt;
      }
      __syncwarp();
      // the spelling node each listed extension leads to
      for (int k = lane; k < KC; k += 32) {
        if (k >= cnt) {
          c_tok[w][k] = -1;
          continue;
        }
        const int tok = c_tok[w][k];
        c_lex[w][k] = tok == d ? 0 : lex_child(lx, ln, tok);
      }
      if (lane == 0) {
        b_lex[w] = ln;
        b_dlm[w] = dlm;
      }
    }
    __syncthreads();

    if (warp == 0) {
      const bool valid = lane < nb;
      s_node[lane] = valid ? node : -2;
      const int par = valid ? tr.parent[node] : -3;
      const int tk = valid ? tr.token[node] : -1;
      __syncwarp();
      int pl = -1;
      if (valid && par >= 0)
        for (int j = 0; j < nb; ++j)
          if (s_node[j] == par) pl = j;
      s_pl[lane] = pl;
      s_tk[lane] = tk;
      s_last[lane] = last;
      s_score[lane] = score;
      __syncwarp();

      double e_score = -INFINITY;
      int e_last = blank;
      long long e_order = kNoOrder;
      bool e_avail = valid;
      if (valid) {
        double cs[3];
        int cl[3];
        long long co[3];
        bool ch[3];
        const bool h1 = pl >= 0 && s_last[pl] != tk;
        const double sc1 =
            h1 ? (tk == d ? word_offer(s_score[pl], lp(tk), b_lex[pl] != 0, b_dlm[pl], lmw, ws) : s_score[pl] + lp(tk))
               : 0.0;
        const long long o1 = (long long)pl * Vp + 1 + tk;
        const bool h3 = last >= 0 && last != blank;
        const double sc3 = h3 ? score + lp(last) : 0.0;
        const int first = (h1 && pl < lane) ? 0 : 2;
        const int i2 = first == 0 ? 1 : 0, i3 = i2 + 1;
        cs[first] = sc1, cl[first] = tk, co[first] = o1, ch[first] = h1;
        cs[i2] = score + lp(blank), cl[i2] = blank, co[i2] = (long long)lane * Vp, ch[i2] = true;
        cs[i3] = sc3, cl[i3] = last, co[i3] = (long long)lane * Vp + 1 + last, ch[i3] = h3;
        bool none = true;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          if (!ch[i]) continue;
          if (none || cs[i] > e_score) {
            e_score = cs[i];
            e_last = cl[i];
          }
          if (none) e_order = co[i];
          none = false;
        }
      }

      int p = valid ? 0 : KC;
      int x_tok = -1;
      double x_score = -INFINITY;
      auto advance = [&]() {
        while (p < KC) {
          const int tok = c_tok[lane][p];
          if (tok < 0) {
            p = KC;
            break;
          }
          bool skip = tok == last;
          for (int j = 0; j < nb && !skip; ++j) skip = s_pl[j] == lane && s_tk[j] == tok;
          if (!skip) {
            x_tok = tok;
            x_score = c_sc[lane][p];
            return;
          }
          ++p;
        }
      };
      advance();

      int count = 0;
      for (int r = 0; r < W; ++r) {
        const bool hx = p < KC;
        const long long x_order = (long long)lane * Vp + 1 + x_tok;
        bool take_e = e_avail;
        if (e_avail && hx) take_e = e_score > x_score || (e_score == x_score && e_order < x_order);
        double ps = take_e ? e_score : (hx ? x_score : -INFINITY);
        long long po = take_e ? e_order : (hx ? x_order : kNoOrder);
        double bs = ps;
        long long bo = po;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const double os = __shfl_xor_sync(0xffffffffu, bs, o);
          const long long oo = __shfl_xor_sync(0xffffffffu, bo, o);
          if (oo != kNoOrder && (bo == kNoOrder || os > bs || (os == bs && oo < bo))) {
            bs = os;
            bo = oo;
          }
        }
        if (bo == kNoOrder) break;
        const bool mine = po == bo;
        bool created = false;
        if (mine) {
          if (take_e) {
            n_node[r] = node;
            n_score[r] = e_score;
            n_last[r] = e_last;
            e_avail = false;
          } else {
            int c = tr.first_child[node];
            while (c >= 0 && tr.token[c] != x_tok) c = tr.next_sibling[c];
            if (c < 0) {
              c = n_nodes;
              tr.parent[c] = node;
              tr.token[c] = x_tok;
              tr.depth[c] = tr.depth[node] + 1;
              tr.first_child[c] = -1;
              tr.next_sibling[c] = tr.first_child[node];
              tr.first_child[node] = c;
              tr.lex[c] = c_lex[lane][p];
              const bool closes = x_tok == d && b_lex[lane] != 0;
              tr.closer[c] = closes ? c : tr.closer[node];
              tr.word[c] = closes ? word_of(lx, b_lex[lane]) : -1;
              tr.nwords[c] = tr.nwords[node] + (closes ? 1 : 0);
              tr.close_lm[c] = __int_as_float(0x7fffffff);
              created = true;
            }
            n_node[r] = c;
            n_score[r] = x_score;
            n_last[r] = x_tok;
            ++p;
            advance();
          }
        }
        n_nodes += __ballot_sync(0xffffffffu, created) != 0;
        ++count;
      }
      __syncwarp();
      nb = count;
      if (lane < nb) {
        node = n_node[lane];
        score = n_score[lane];
        last = n_last[lane];
        b_node[lane] = node;
        b_score[lane] = score;
      }
      if (lane == 0) b_nb = nb;
    }
    __syncthreads();
  }

  if (warp == 0) {
    // end of utterance: close the pending run, add </s>, stable sort
    bool keep = lane < nb;
    double f = -INFINITY;
    if (keep) {
      const int ln = tr.lex[node];
      int extra = -1;
      f = score;
      if (ln != 0) {
        if (lx.constrained && (ln < 0 || lx.word[ln] < 0)) {
          keep = false;
        } else {
          extra = word_of(lx, ln);
          f = __dadd_rn(__dadd_rn(f, __dmul_rn(lmw, (double)word_lm(lm, tr, node, -1, extra))), ws);
        }
      }
      if (keep) f = __dadd_rn(f, __dmul_rn(lmw, (double)word_lm(lm, tr, node, extra, lx.eos)));
    }
    n_score[lane] = f;
    n_node[lane] = keep;
    __syncwarp();
    const unsigned keepm = __ballot_sync(0xffffffffu, keep);
    const int cnt = __popc(keepm);
    int rank = 0;
    for (int j = 0; j < nb; ++j)
      if (n_node[j] && (n_score[j] > f || (n_score[j] == f && j < lane))) ++rank;
    if (keep) {
      int32_t* out = out_tokens + (b * W + rank) * L;
      const int len = tr.depth[node];
      out_scores[b * W + rank] = f;
      out_lens[b * W + rank] = len;
      int nd = node;
      for (int i = len - 1; i >= 0; --i) {
        out[i] = tr.token[nd];
        nd = tr.parent[nd];
      }
      for (int64_t i = len; i < L; ++i) out[i] = -1;
    }
    if (lane >= cnt && lane < W) {
      int32_t* out = out_tokens + (b * W + lane) * L;
      out_scores[b * W + lane] = -INFINITY;
      out_lens[b * W + lane] = -1;
      for (int64_t i = 0; i < L; ++i) out[i] = -1;
    }
  }
}

}  // namespace

cudaError_t launch_beam_rows(const float* logits, float2* stats, int32_t* top_tok, int64_t M, int V, int K,
                             int blank, int64_t L, const int32_t* lens, int lens_stride, cudaStream_t s,
                             int64_t* launches) {
  if (M <= 0) return cudaSuccess;
  beam_rows_kernel<<<(unsigned)((M + 7) / 8), 256, 0, s>>>(logits, stats, top_tok, M, V, K, blank, L, lens,
                                                           lens_stride);
  if (launches) ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_beam_search(const float* logits, const float2* stats, const int32_t* top_tok, int K, int64_t B,
                               int64_t L, const int32_t* lens, int lens_stride, int V, int W, int blank,
                               int32_t* trie, int64_t trie_cap, int32_t* out_tokens, int32_t* out_lens,
                               double* out_scores, cudaStream_t s, int64_t* launches) {
  if (B <= 0) return cudaSuccess;
  beam_search_kernel<<<(unsigned)B, 32, 0, s>>>(logits, stats, top_tok, K, L, lens, lens_stride, V, W, blank, trie,
                                                trie + B * trie_cap, trie + 2 * B * trie_cap, trie_cap, out_tokens,
                                                out_lens, out_scores);
  if (launches) ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_beam_search_lm(const float* logits, const float2* stats, const LmView& lm, double lm_weight,
                                  int64_t B, int64_t L, const int32_t* lens, int lens_stride, int V, int W, int blank,
                                  int32_t* trie, float* trie_lm, int64_t trie_cap, float* rows, int32_t* out_tokens,
                                  int32_t* out_lens, double* out_scores, cudaStream_t s) {
  if (B <= 0) return cudaSuccess;
  const int K = V - 1 < W + 1 ? (V - 1 > 0 ? V - 1 : 1) : W + 1;
  const int warps = W < 16 ? W : 16;
  beam_search_lm_kernel<<<(unsigned)B, 32 * warps, 0, s>>>(logits, stats, lm, lm_weight, K, L, lens, lens_stride, V,
                                                           W, blank, trie, trie + B * trie_cap,
                                                           trie + 2 * B * trie_cap, trie + 3 * B * trie_cap,
                                                           trie + 4 * B * trie_cap, trie_lm, trie_cap, rows,
                                                           out_tokens, out_lens, out_scores);
  return cudaGetLastError();
}

cudaError_t launch_beam_search_word_lm(const float* logits, const float2* stats, const int32_t* top_tok, int K,
                                       const LmView& lm, const LexView& lx, double lm_weight, double word_score,
                                       int64_t B, int64_t L, const int32_t* lens, int lens_stride, int V, int W,
                                       int blank, int32_t* trie, float* trie_f, int64_t trie_cap, int32_t* out_tokens,
                                       int32_t* out_lens, double* out_scores, cudaStream_t s) {
  if (B <= 0) return cudaSuccess;
  const int warps = W < 16 ? W : 16;
  beam_search_word_lm_kernel<<<(unsigned)B, 32 * warps, 0, s>>>(logits, stats, top_tok, K, lm, lx, lm_weight,
                                                                word_score, L, lens, lens_stride, V, W, blank, trie,
                                                                trie_f, trie_cap, out_tokens, out_lens, out_scores);
  return cudaGetLastError();
}

}  // namespace vasr
