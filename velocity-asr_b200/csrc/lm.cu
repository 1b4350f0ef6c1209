// lm.cu — ARPA n-gram language models over token ids or over words: the host parser (validation before any device call), the
// upload of the device tables (layout: lm.cuh) and the scoring kernel behind vasr_lm_log_prob.
//
// Vocabulary mapping: an ARPA word maps to the vocabulary entry with the same string (the first one), the word
// <space> to the entry " ".  <s> is the context symbol V and only a context: an n-gram with <s> anywhere but first,
// or with a word outside the vocabulary (</s> included), can never be reached and is dropped.  Duplicate lines:
// the last one wins.
// A word LM (lm_parse_word_arpa) is the same parse over the file's own unigram words instead of a vocabulary, plus
// the spelling trie of its lexicon over the token ids of the character vocabulary.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string_view>
#include <unordered_map>

#include "common.cuh"
#include "lm.cuh"

namespace vasr {

namespace {

constexpr int kMaxFields = kLmMaxOrder + 2;   // log-prob, up to 8 words, back-off weight

struct Entry {
  int32_t node, tok;
  float lp;
};

bool is_ws(char c) { return c == ' ' || c == '\t' || c == '\r'; }

// ARPA values are log10: parsed as fp64, times ln 10 in fp64, rounded once to fp32
bool parse_log10(std::string_view f, float* out) {
  if (f.empty()) return false;
  char* end = nullptr;
  const double v = strtod(f.data(), &end);   // the buffer is NUL-terminated and a field ends at white space
  if (end != f.data() + f.size() || !std::isfinite(v)) return false;
  *out = (float)(v * M_LN10);
  return true;
}

bool parse_count(std::string_view f, int64_t* out) {
  if (f.empty() || f.size() > 18) return false;
  int64_t v = 0;
  for (char c : f) {
    if (c < '0' || c > '9') return false;
    v = v * 10 + (c - '0');
  }
  *out = v;
  return true;
}

// "\N-grams:" -> N, else 0
int section_order(std::string_view f) {
  const std::string_view tail = "-grams:";
  if (f.size() < 2 + tail.size() || f[0] != '\\' || f.substr(f.size() - tail.size()) != tail) return 0;
  int64_t n = 0;
  if (!parse_count(f.substr(1, f.size() - 1 - tail.size()), &n) || n < 1 || n > 1000) return 0;
  return (int)n;
}

bool read_file(const char* path, std::string* buf) {
  FILE* fp = fopen(path, "rb");
  if (!fp) return false;
  char chunk[1 << 16];
  size_t n;
  while ((n = fread(chunk, 1, sizeof chunk, fp)) > 0) buf->append(chunk, n);
  fclose(fp);
  return true;
}

}  // namespace

bool lm_parse_arpa(const char* path, const char* const* vocab, int V, int blank, LmHostTables* t, std::string* err) {
  const std::string where = std::string(path);
  auto fail_at = [&](int64_t line, const std::string& msg) {
    *err = where + ", line " + std::to_string(line) + ": " + msg;
    return false;
  };
  std::string buf;
  if (!read_file(path, &buf)) {
    *err = where + ": cannot open";
    return false;
  }

  std::unordered_map<std::string_view, int> word_id;
  word_id.reserve((size_t)V * 2);
  for (int i = 0; i < V; ++i) {
    if (!vocab[i]) {
      *err = "vocabulary entry " + std::to_string(i) + " is NULL";
      return false;
    }
    const std::string_view w(vocab[i]);
    word_id.emplace(w == " " ? std::string_view("<space>") : w, i);
  }

  // context trie over reversed histories, built on the fly
  std::unordered_map<unsigned long long, int32_t> child;
  std::vector<float> bow(1, 0.f);
  auto node_of = [&](const int32_t* ids, int q) {   // context ids[0 .. q), newest last
    int32_t c = 0;
    for (int i = q - 1; i >= 0; --i) {
      const unsigned long long key = ((unsigned long long)(unsigned)c << 32) | (unsigned)ids[i];
      auto it = child.find(key);
      if (it == child.end()) {
        const int32_t nc = (int32_t)bow.size();
        bow.push_back(0.f);
        it = child.emplace(key, nc).first;
      }
      c = it->second;
    }
    return c;
  };
  std::vector<Entry> entries;
  std::vector<float> uni_listed((size_t)V, 0.f);
  std::vector<char> uni_has((size_t)V, 0);
  bool has_unk = false;
  float unk = 0.f;

  std::vector<int64_t> counts;
  int stage = 0;            // 0: before the data line, 1: counts, 2: between sections, 3: in section `cur`, 4: done
  int cur = 0, order = 0;
  int64_t seen = 0, line = 0, uni_line = 0;
  const char* p = buf.data();
  const char* const e = p + buf.size();
  while (p < e && stage != 4) {
    const char* nl = static_cast<const char*>(memchr(p, '\n', (size_t)(e - p)));
    const char* le = nl ? nl : e;
    ++line;
    std::string_view f[kMaxFields];
    int nf = 0;
    bool too_many = false;
    for (const char* q = p; q < le;) {
      while (q < le && is_ws(*q)) ++q;
      if (q >= le) break;
      const char* s = q;
      while (q < le && !is_ws(*q)) ++q;
      if (nf < kMaxFields) f[nf++] = std::string_view(s, (size_t)(q - s));
      else too_many = true;
    }
    p = nl ? nl + 1 : e;
    if (nf == 0) continue;

    if (stage == 3 && f[0][0] == '\\') {
      if (seen != counts[cur - 1])
        return fail_at(line, "the " + std::to_string(cur) + "-gram section has " + std::to_string(seen) +
                                 " entries, \\data\\ says " + std::to_string(counts[cur - 1]));
      stage = 2;
    }
    switch (stage) {
      case 0:
        if (nf == 1 && f[0] == "\\data\\") stage = 1;
        break;
      case 1: {
        if (nf == 2 && f[0] == "ngram") {
          const size_t eq = f[1].find('=');
          int64_t n = 0, c = 0;
          if (eq == std::string_view::npos || !parse_count(f[1].substr(0, eq), &n) ||
              !parse_count(f[1].substr(eq + 1), &c))
            return fail_at(line, "bad \\data\\ line");
          if (n != (int64_t)counts.size() + 1) return fail_at(line, "\\data\\ counts must list orders 1, 2, ... in turn");
          if (n > kLmMaxOrder) return fail_at(line, "order " + std::to_string(n) + " is above 8");
          counts.push_back(c);
          break;
        }
        if (counts.empty()) return fail_at(line, "bad header: expected `ngram 1=<count>` after \\data\\");
        order = (int)counts.size();
        stage = 2;
      }
        [[fallthrough]];
      case 2: {
        if (nf == 1 && f[0] == "\\end\\") {
          if (cur != order)
            return fail_at(line, "\\end\\ before the " + std::to_string(cur + 1) + "-gram section");
          stage = 4;
          break;
        }
        const int n = nf == 1 ? section_order(f[0]) : 0;
        if (n != cur + 1 || n > order)
          return fail_at(line, "expected \\" + std::to_string(cur + 1) + "-grams: or \\end\\");
        cur = n;
        seen = 0;
        if (n == 1) uni_line = line;
        stage = 3;
        break;
      }
      case 3: {
        const int n = cur;
        if (++seen > counts[n - 1])
          return fail_at(line, "more " + std::to_string(n) + "-grams than \\data\\ says (" +
                                   std::to_string(counts[n - 1]) + ")");
        if (too_many || !(nf == n + 1 || (nf == n + 2 && n < order)))
          return fail_at(line, "a " + std::to_string(n) + "-gram line has a log-prob, " + std::to_string(n) +
                                   " words" + (n < order ? " and an optional back-off weight" : ""));
        float lp = 0.f, bw = 0.f;
        if (!parse_log10(f[0], &lp)) return fail_at(line, "unparsable number `" + std::string(f[0]) + "`");
        if (nf == n + 2 && !parse_log10(f[n + 1], &bw))
          return fail_at(line, "unparsable number `" + std::string(f[n + 1]) + "`");
        if (n == 1 && f[1] == "<unk>") {
          has_unk = true;
          unk = lp;
        }
        int32_t ids[kLmMaxOrder] = {};
        bool keep = true;
        for (int i = 0; i < n && keep; ++i) {
          if (f[1 + i] == "<s>") {
            ids[i] = V;
            keep = i == 0;
          } else {
            auto it = word_id.find(f[1 + i]);
            keep = it != word_id.end();
            ids[i] = keep ? it->second : -1;
          }
        }
        if (!keep) break;
        ++t->kept;
        if (ids[n - 1] != V) {
          if (n == 1) {
            uni_listed[ids[0]] = lp;
            uni_has[ids[0]] = 1;
          } else {
            entries.push_back({node_of(ids, n - 1), ids[n - 1], lp});
          }
        }
        if (n < order) bow[node_of(ids, n)] = bw;
        break;
      }
    }
  }
  if (stage == 0) return fail_at(line + 1, "bad header: no \\data\\ line");
  if (stage == 3 && seen != counts[cur - 1])
    return fail_at(line + 1, "the " + std::to_string(cur) + "-gram section has " + std::to_string(seen) +
                                 " entries, \\data\\ says " + std::to_string(counts[cur - 1]));
  if (stage != 4) return fail_at(line + 1, "missing \\end\\");

  t->order = order;
  t->V = V;
  t->listed = 0;
  for (int64_t c : counts) t->listed += c;
  t->uni.resize((size_t)V);
  for (int i = 0; i < V; ++i) {
    if (uni_has[i]) t->uni[i] = uni_listed[i];
    else if (has_unk) t->uni[i] = unk;
    else if (i == blank) t->uni[i] = -INFINITY;   // never scored
    else
      return fail_at(uni_line, "token " + std::to_string(i) + " (`" + vocab[i] +
                                   "`) has no unigram and the file has no <unk>");
  }

  // CSR of continuations per context node, token ascending, the last duplicate kept
  std::stable_sort(entries.begin(), entries.end(),
                   [](const Entry& a, const Entry& b) { return a.node != b.node ? a.node < b.node : a.tok < b.tok; });
  const int64_t nodes = (int64_t)bow.size();
  t->off.assign((size_t)nodes + 1, 0);
  t->cont_tok.clear();
  t->cont_lp.clear();
  t->cont_tok.reserve(entries.size());
  t->cont_lp.reserve(entries.size());
  for (size_t i = 0; i < entries.size(); ++i) {
    if (i + 1 < entries.size() && entries[i + 1].node == entries[i].node && entries[i + 1].tok == entries[i].tok)
      continue;
    t->cont_tok.push_back(entries[i].tok);
    t->cont_lp.push_back(entries[i].lp);
    ++t->off[(size_t)entries[i].node + 1];
  }
  for (int64_t n = 0; n < nodes; ++n) t->off[n + 1] += t->off[n];
  t->bow = std::move(bow);

  // open-addressing child table, at most half full
  int64_t cap = 2;
  while (cap < 2 * (int64_t)child.size()) cap <<= 1;
  t->hash_key.assign((size_t)cap, kLmEmpty);
  t->hash_val.assign((size_t)cap, -1);
  for (const auto& kv : child) {
    unsigned long long h = lm_hash(kv.first) & (unsigned long long)(cap - 1);
    while (t->hash_key[h] != kLmEmpty) h = (h + 1) & (unsigned long long)(cap - 1);
    t->hash_key[h] = kv.first;
    t->hash_val[h] = kv.second;
  }
  return true;
}

cudaError_t lm_upload(const LmHostTables& t, void** block, LmView* view) {
  const size_t sizes[7] = {t.hash_key.size() * 8, t.hash_val.size() * 4, t.bow.size() * 4, t.off.size() * 8,
                           t.cont_tok.size() * 4, t.cont_lp.size() * 4, t.uni.size() * 4};
  const void* src[7] = {t.hash_key.data(), t.hash_val.data(), t.bow.data(), t.off.data(),
                        t.cont_tok.data(), t.cont_lp.data(), t.uni.data()};
  size_t at[7], total = 0;
  for (int i = 0; i < 7; ++i) {
    at[i] = total;
    total += (sizes[i] + 255) / 256 * 256;
  }
  char* base = nullptr;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&base), total > 0 ? total : 256);
  if (e != cudaSuccess) return e;
  for (int i = 0; i < 7; ++i) {
    if (sizes[i] == 0) continue;
    e = cudaMemcpy(base + at[i], src[i], sizes[i], cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      cudaFree(base);
      return e;
    }
  }
  *block = base;
  view->order = t.order;
  view->V = t.V;
  view->hash_cap = (int64_t)t.hash_key.size();
  view->hash_key = reinterpret_cast<const unsigned long long*>(base + at[0]);
  view->hash_val = reinterpret_cast<const int32_t*>(base + at[1]);
  view->bow = reinterpret_cast<const float*>(base + at[2]);
  view->off = reinterpret_cast<const int64_t*>(base + at[3]);
  view->cont_tok = reinterpret_cast<const int32_t*>(base + at[4]);
  view->cont_lp = reinterpret_cast<const float*>(base + at[5]);
  view->uni = reinterpret_cast<const float*>(base + at[6]);
  return cudaSuccess;
}

bool lm_parse_word_arpa(const char* path, const char* const* vocab, int V, int blank, const char* delimiter,
                        bool constrained, LmHostTables* t, LexHostTables* x, std::string* err) {
  for (int i = 0; i < V; ++i)
    if (!vocab[i]) {
      *err = "vocabulary entry " + std::to_string(i) + " is NULL";
      return false;
    }
  x->delim = -1;
  for (int i = 0; i < V && x->delim < 0; ++i)
    if (strcmp(vocab[i], delimiter) == 0) x->delim = i;
  if (x->delim < 0) {
    *err = std::string("the word delimiter `") + delimiter + "` is not in the vocabulary";
    return false;
  }
  if (x->delim == blank) {
    *err = std::string("the word delimiter `") + delimiter + "` is the blank token (" + std::to_string(blank) + ")";
    return false;
  }

  // the words: the unigram section's, <s> excluded, first occurrence first; lm_parse_arpa then takes them as its
  // vocabulary, so word id = index and <s> is the context symbol as for a token LM
  std::string buf;
  if (!read_file(path, &buf)) {
    *err = std::string(path) + ": cannot open";
    return false;
  }
  {
    std::unordered_map<std::string_view, int> seen;
    bool in_uni = false;
    int64_t line = 0, uni_line = 0;
    const char* p = buf.data();
    const char* const e = p + buf.size();
    while (p < e) {
      const char* nl = static_cast<const char*>(memchr(p, '\n', (size_t)(e - p)));
      const char* le = nl ? nl : e;
      ++line;
      std::string_view f[2];
      int nf = 0;
      for (const char* q = p; q < le && nf < 2;) {
        while (q < le && is_ws(*q)) ++q;
        if (q >= le) break;
        const char* s = q;
        while (q < le && !is_ws(*q)) ++q;
        f[nf++] = std::string_view(s, (size_t)(q - s));
      }
      p = nl ? nl + 1 : e;
      if (nf == 0) continue;
      if (in_uni && f[0][0] == '\\') break;
      if (f[0] == "\\1-grams:") {
        in_uni = true;
        uni_line = line;
      } else if (in_uni && nf == 2 && f[1] != "<s>" && seen.emplace(f[1], (int)x->words.size()).second) {
        x->words.emplace_back(f[1]);
      }
    }
    std::vector<const char*> names(x->words.size());
    for (size_t i = 0; i < names.size(); ++i) names[i] = x->words[i].c_str();
    if (!lm_parse_arpa(path, names.data(), (int)names.size(), -1, t, err)) return false;
    auto id = [&](const char* w) {
      auto it = seen.find(w);
      return it == seen.end() ? -1 : it->second;
    };
    x->unk = id("<unk>");
    x->eos = id("</s>") >= 0 ? id("</s>") : x->unk;
    const std::string at = std::string(path) + ", line " + std::to_string(uni_line) + ": ";
    if (!constrained && x->unk < 0) {
      *err = at + "lexicon-free mode needs <unk> (a word outside the lexicon scores as <unk>); the file has none";
      return false;
    }
    if (x->eos < 0) {
      *err = at + "the file has neither </s> nor <unk> to score the end of an utterance";
      return false;
    }
  }

  // spelling: one token per character (UTF-8 code point), the first vocabulary entry with that string, which must
  // be neither the blank nor the delimiter
  std::unordered_map<std::string_view, int> char_tok;
  for (int i = V - 1; i >= 0; --i) char_tok[std::string_view(vocab[i])] = i;   // the first entry wins
  std::vector<std::map<int32_t, int32_t>> kids(1);
  std::vector<int32_t> word_at(1, -1);
  x->lexicon = 0;
  std::vector<int32_t> spell;
  for (size_t w = 0; w < x->words.size(); ++w) {
    const std::string& s = x->words[w];
    if (s == "<unk>" || s == "</s>") continue;
    spell.clear();
    bool ok = !s.empty();
    for (size_t i = 0; i < s.size() && ok;) {
      const unsigned char c = (unsigned char)s[i];
      const size_t n = c < 0x80 ? 1 : (c & 0xe0) == 0xc0 ? 2 : (c & 0xf0) == 0xe0 ? 3 : (c & 0xf8) == 0xf0 ? 4 : 1;
      auto it = char_tok.find(std::string_view(s).substr(i, n));
      ok = it != char_tok.end() && it->second != blank && it->second != x->delim;
      if (ok) spell.push_back(it->second);
      i += n;
    }
    if (!ok) continue;
    int32_t node = 0;
    for (int32_t tk : spell) {
      auto it = kids[node].find(tk);
      if (it == kids[node].end()) {
        it = kids[node].emplace(tk, (int32_t)kids.size()).first;
        kids.emplace_back();
        word_at.push_back(-1);
      }
      node = it->second;
    }
    word_at[node] = (int32_t)w;
    ++x->lexicon;
  }
  if (constrained && x->lexicon == 0) {
    *err = "lexicon-constrained mode needs a lexicon: none of the file's " + std::to_string(x->words.size()) +
           " words can be spelled in the vocabulary";
    return false;
  }
  x->off.assign(kids.size() + 1, 0);
  x->tok.clear();
  x->child.clear();
  for (size_t n = 0; n < kids.size(); ++n) {
    for (const auto& kv : kids[n]) {
      x->tok.push_back(kv.first);
      x->child.push_back(kv.second);
    }
    x->off[n + 1] = (int32_t)x->tok.size();
  }
  x->word = std::move(word_at);
  return true;
}

cudaError_t lex_upload(const LexHostTables& x, bool constrained, void** block, LexView* view) {
  const std::vector<int32_t>* parts[4] = {&x.off, &x.tok, &x.child, &x.word};
  size_t at[4], total = 0;
  for (int i = 0; i < 4; ++i) {
    at[i] = total;
    total += (parts[i]->size() * 4 + 255) / 256 * 256;
  }
  char* base = nullptr;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&base), total > 0 ? total : 256);
  if (e != cudaSuccess) return e;
  for (int i = 0; i < 4; ++i) {
    if (parts[i]->empty()) continue;
    e = cudaMemcpy(base + at[i], parts[i]->data(), parts[i]->size() * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
      cudaFree(base);
      return e;
    }
  }
  *block = base;
  view->delim = x.delim;
  view->constrained = constrained ? 1 : 0;
  view->unk = x.unk;
  view->eos = x.eos;
  view->off = reinterpret_cast<const int32_t*>(base + at[0]);
  view->tok = reinterpret_cast<const int32_t*>(base + at[1]);
  view->child = reinterpret_cast<const int32_t*>(base + at[2]);
  view->word = reinterpret_cast<const int32_t*>(base + at[3]);
  return cudaSuccess;
}

namespace {

// one thread per row: the longest listed context that lists the token, then the back-off weights above it
__global__ void __launch_bounds__(256) lm_log_prob_kernel(LmView lm, const int32_t* __restrict__ prefixes,
                                                          const int32_t* __restrict__ lens, int64_t n,
                                                          const int32_t* __restrict__ tokens,
                                                          float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int H = lm.order > 1 ? lm.order - 1 : 1;
  const int32_t* pre = prefixes + i * H;
  const int len = lens[i], tok = tokens[i];
  if (tok < 0 || tok >= lm.V || len < 0) {
    out[i] = __int_as_float(0x7fffffff);
    return;
  }
  const int k = min(lm.order - 1, len + 1);
  out[i] = lm_score(lm, k, [&](int q) { return q <= len ? pre[H - q] : lm.V; }, tok);
}

}  // namespace

cudaError_t launch_lm_log_prob(const LmView& lm, const int32_t* prefixes, const int32_t* lens, int64_t n,
                               const int32_t* tokens, float* out, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  lm_log_prob_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(lm, prefixes, lens, n, tokens, out);
  return cudaGetLastError();
}

}  // namespace vasr
