// engine.cu — the C ABI of libvasr.so (include/vasr.h): handle, weight intake and packing,
// workspace arena, and the launch sequence of the VELOCITY-ASR v2 inference path
//   PCM -> log-mel -> temporal binding -> 8 SSM blocks -> global context -> CTC head -> greedy
// (scripts/transcribe.py:69-82 -> audio.py:65 -> model.py:333-368 -> decode.py:27).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/vasr.h"
#include "common.cuh"
#include "kernels.cuh"
#include "lm.cuh"

using namespace vasr;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CK(expr)                                                                               \
  do {                                                                                         \
    cudaError_t e_ = (expr);                                                                   \
    if (e_ != cudaSuccess)                                                                     \
      return fail(VASR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_) + " (" +   \
                                     __FILE__ + ":" + std::to_string(__LINE__) + ")");         \
  } while (0)

#define RET(expr)            \
  do {                       \
    int r_ = (expr);         \
    if (r_ != VASR_OK) return r_; \
  } while (0)

constexpr int N_FFT = 400, HOP = 160, N_FREQ = 201, PAD = 200;

struct BlockW {
  float *ln1_g, *ln1_b, *ln2_g, *ln2_b, *conv_w, *conv_b, *A, *D;
  float *w_in, *w_xdt, *b_xdt, *w_out, *w_f1, *b_f1, *w_f2, *b_f2;
  float* s_f1;             // norm2 is folded into ffn.0 (fold_ln): column sums of the folded weight
  int N = 0;
  int di = 0, ks = 0;      // d_inner and depthwise kernel size of THIS stack (GlobalSSM hard-codes 2 / 4: ssm.py:529-538)
  int structured = 0;
};

// One projection that hosts FakeQuantize'd reference modules (config 5): per-column output scale / zero
// point on the device, and which column ranges belong to which module (quantize.py:142-191, 194-266).
struct QSite {
  float *qs = nullptr, *qz = nullptr;   // (N) device; scale <= 0 -> column not quantised / not calibrated
  int N = 0;
  int nmod = 0;
  const char* name[3] = {nullptr, nullptr, nullptr};
  int c0[3] = {0, 0, 0}, nc[3] = {0, 0, 0};
};
enum { Q_TB = 0, Q_P1, Q_P2, Q_Q, Q_KV, Q_O, Q_F3, Q_FO, Q_CTC, Q_SITES };

struct Arena {
  char* base = nullptr;
  size_t bytes = 0;
  size_t used = 0;
  void reset() { used = 0; }
  template <typename T>
  T* take(int64_t n) {
    size_t off = (used + 255) & ~size_t(255);
    used = off + (size_t)(n > 0 ? n : 0) * sizeof(T);
    return reinterpret_cast<T*>(base + off);
  }
};

}  // namespace

struct vasr_handle {
  vasr_config cfg{};
  int device = 0;
  std::unordered_map<std::string, std::vector<float>> staged;
  bool committed = false;
  std::vector<void*> weight_allocs;
  std::vector<void*> frontend_allocs;
  std::vector<void*>* alloc_list = &weight_allocs;
  // config 5: FakeQuantize of the 12 non-SSM modules (quantize.py:269-322 with ssm_state_fp32)
  int quant = 0;             // requested; applied at commit
  int quant_active = 0;      // the committed weights are fake-quantised and the sites below exist
  int calibrating = 0;       // this forward updates the activation scales before using them
  QSite qsite[Q_SITES];
  // pinned staging of a ragged batch's per-utterance dims: a ring, so a call never waits for the stream unless
  // all RAG_RING earlier uploads are still queued
  static constexpr int RAG_RING = 4;
  int32_t* rag_pin[RAG_RING] = {};
  cudaEvent_t rag_ev[RAG_RING] = {};
  int64_t rag_pin_cap = 0;
  int rag_next = 0;
  float* q_mm = nullptr;     // (2) min / max scratch
  // TF32 hi/lo split of each weight matrix the tensor-core kernel has used, keyed by the fp32 copy
  std::unordered_map<const float*, float*> w_split;

  std::vector<BlockW> local, global;
  float *tb_w = nullptr, *tb_b = nullptr, *pe_time = nullptr, *pe_freq = nullptr, *tb_g = nullptr, *tb_bt = nullptr;
  int64_t pe_rows = 0;
  float *loc_g = nullptr, *loc_b = nullptr, *glo_g = nullptr, *glo_b = nullptr;
  float *p1_w = nullptr, *p1_b = nullptr, *p2_w = nullptr, *p2_b = nullptr;
  float *n1_g = nullptr, *n1_b = nullptr, *n2_g = nullptr, *n2_b = nullptr;
  float *w_q = nullptr, *b_q = nullptr, *w_kv = nullptr, *b_kv = nullptr, *w_o = nullptr, *b_o = nullptr;
  float *w_f3 = nullptr, *b_f3 = nullptr, *w_fo = nullptr, *b_fo = nullptr;
  float *ctc_g = nullptr, *ctc_b = nullptr, *w_ctc = nullptr, *b_ctc = nullptr;
  // fp32 model only (the FakeQuantize model keeps its modules one by one, quantize.py:269-322): LayerNorms folded
  // into the projection that follows them (fold_ln), and the fusion's stacked projection with its rows permuted for
  // the gate epilogue (gate_perm_row)
  float *w_q_ln = nullptr, *b_q_ln = nullptr, *s_q = nullptr, *w_kv_ln = nullptr, *b_kv_ln = nullptr, *s_kv = nullptr;
  float *w_ctc_ln = nullptr, *b_ctc_ln = nullptr, *s_ctc = nullptr, *w_f3p = nullptr, *b_f3p = nullptr;
  float* win = nullptr;      // analysis window (400)
  float* tw400 = nullptr;    // W400^m = (cos, -sin)(2 pi m / 400)
  int *fb_lo = nullptr, *fb_off = nullptr;
  float* fb_w = nullptr;

  int num_sms = 148;
  int64_t tc_launches = 0;

  Arena ws;
  cudaStream_t own_stream = nullptr;
  // host entry points: the PCM travels in HOST_SLICES pieces on copy_stream, the log-mel of a piece starts when it
  // has landed (the mel is per utterance), so the front end runs under the tail of the transfer
  static constexpr int HOST_SLICES = 8;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t slice_ev[HOST_SLICES] = {};
  cudaEvent_t copy_gate = nullptr;
  int64_t launches = 0;
  // Calls on one handle share the workspace and the lazily built weight splits.  Each call leaves an event at
  // its end on its stream; a call arriving on ANOTHER stream (the *_host entry points use own_stream) waits for
  // it on the device before touching either, so an asynchronous forward followed by a host transcribe is ordered.
  cudaEvent_t call_done = nullptr;
  cudaStream_t call_stream = nullptr;
  bool call_pending = false;

  // VASR_PROF=1: CUDA-event pairs around every projection launch, aggregated by shape (tools/gemm_profile.py)
  int prof = 0;
  struct ProfEntry { std::string tag; cudaEvent_t e0, e1; };
  std::vector<ProfEntry> prof_ev;
  // timing of the scan launches inside the last transcribe/forward
  bool timing = false;
  std::vector<cudaEvent_t> ev;   // pairs
  int ev_used = 0;
  cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
  bool ev_total = false;
};

namespace {

struct Dims {
  int64_t B, S, T, L, M, K1, K2, Mg, M2, Tp;
  int d, di, n_mels, V, att;
};

// GlobalSSM is built with expand_ratio = 2 and kernel_size = 4 whatever the config says (ssm.py:529-538)
constexpr int GLOBAL_EXPAND = 2, GLOBAL_KS = 4;

Dims make_dims(const vasr_handle* h, int64_t B, int64_t S, int64_t T) {
  Dims q{};
  q.B = B;
  q.S = S;
  q.T = T;
  q.L = (T + 1) / 2;
  q.M = B * q.L;
  int64_t k1 = q.L / 8 > 64 ? q.L / 8 : 64;
  q.K1 = k1 < q.L ? k1 : q.L;
  int64_t k2 = q.K1 / 4 > 16 ? q.K1 / 4 : 16;
  k2 = k2 < 64 ? k2 : 64;
  q.K2 = k2 < q.K1 ? k2 : q.K1;
  q.Mg = B * q.K1;
  q.M2 = B * q.K2;
  q.Tp = T + 2 + ((T + 2) & 1);                       // even: batch stride is a multiple of the 2-frame row stride
  q.d = h->cfg.d_model;
  // widest d_inner of the two stacks: sizes the buffers both share
  q.di = h->cfg.d_model * (h->cfg.ssm_expand_ratio > GLOBAL_EXPAND ? h->cfg.ssm_expand_ratio : GLOBAL_EXPAND);
  q.n_mels = h->cfg.mel_bins;
  q.V = h->cfg.vocab_size;
  q.att = h->cfg.attention_dim;
  return q;
}

struct Work {
  float *raw, *melpad;
  double* part;
  float* qscratch;      // probe output of a quantised projection during calibration (M x max N)
  float *xa, *xb, *u, *xz, *bcdt, *yg, *hbuf, *cat, *f3, *fm, *fused, *qb, *ob;
  float *ga, *gb, *g2, *g2n, *kv;
  float* logits;
  float* lnstat;         // (M, 2) row statistics of a projection with a folded LayerNorm
  float* amax_val;       // argmax partials of the CTC head (argmax_slots(V) x M), greedy decode without logits
  int32_t* amax_idx;
  int32_t* pred;
  float* pcm_stage;      // device copies for the *_host entry points
  int32_t *tok_stage, *len_stage;
  int32_t* ragbuf;       // B x RAG_STRIDE per-utterance dims of a ragged batch (kernels.cuh)
  const int32_t* rag;    // = ragbuf for a ragged call, NULL otherwise
};

// Carves the arena; with measure_only it just computes the size.
size_t carve(vasr_handle* h, const Dims& q, bool need_mel, bool need_logits, Work* w, bool need_stage = false) {
  Arena a = h->ws;
  a.reset();
  Work t{};
  const int nmax = h->cfg.ssm_state_dim > h->cfg.global_ssm_state_dim ? h->cfg.ssm_state_dim
                                                                      : h->cfg.global_ssm_state_dim;
  if (need_mel) {
    t.part = a.take<double>(q.B * mel_fft_blocks(q.T) * q.n_mels * 2);
    t.raw = a.take<float>(q.B * q.T * q.n_mels);
  }
  t.melpad = a.take<float>(q.B * q.Tp * q.n_mels);
  t.xa = a.take<float>(q.M * q.d);
  t.xb = a.take<float>(q.M * q.d);
  t.u = a.take<float>(q.M * q.d);
  t.xz = a.take<float>(q.M * 2 * q.di);
  t.bcdt = a.take<float>(q.M * (2 * nmax + q.di));
  t.yg = a.take<float>(q.M * q.di);
  t.hbuf = a.take<float>(q.M * q.di);
  t.cat = a.take<float>(q.M * 2 * q.d);
  if (!h->w_f3p) t.f3 = a.take<float>(q.M * 3 * q.d);      // gate | local | global before gate_mix: only without the gate epilogue
  t.fm = a.take<float>(q.M * q.d);
  t.fused = a.take<float>(q.M * q.d);
  t.qb = a.take<float>(q.M * q.att);
  t.ob = a.take<float>(q.M * q.att);
  t.ga = a.take<float>(q.Mg * q.d);
  t.gb = a.take<float>(q.Mg * q.d);
  t.g2 = a.take<float>(q.M2 * q.d);
  t.g2n = a.take<float>(q.M2 * q.d);
  t.kv = a.take<float>(q.M2 * 2 * q.att);
  if (need_logits) t.logits = a.take<float>(q.M * q.V);
  t.lnstat = a.take<float>(q.M * 2);
  t.amax_val = a.take<float>(q.M * argmax_slots(q.V));
  t.amax_idx = a.take<int32_t>(q.M * argmax_slots(q.V));
  if (h->quant_active) t.qscratch = a.take<float>(q.M * (q.V > 3 * q.d ? q.V : 3 * q.d));
  t.pred = a.take<int32_t>(q.M);
  t.ragbuf = a.take<int32_t>(q.B * RAG_STRIDE);
  if (need_stage) {
    t.pcm_stage = a.take<float>(q.B * q.S);
    t.tok_stage = a.take<int32_t>(q.M);
    t.len_stage = a.take<int32_t>(q.B);
  }
  if (w) *w = t;
  return a.used + 256;
}

int ensure_workspace(vasr_handle* h, const Dims& q, bool need_mel, bool need_logits, Work* w,
                     bool need_stage = false) {
  const size_t need = carve(h, q, need_mel, need_logits, nullptr, need_stage);
  if (need > h->ws.bytes) {
    CK(cudaDeviceSynchronize());
    if (h->ws.base) CK(cudaFree(h->ws.base));
    h->ws.base = nullptr;
    h->ws.bytes = 0;
    void* p = nullptr;
    CK(cudaMalloc(&p, need));
    h->ws.base = static_cast<char*>(p);
    h->ws.bytes = need;
  }
  carve(h, q, need_mel, need_logits, w, need_stage);
  return VASR_OK;
}

// ---------------------------------------------------------------- weights ---------------
const std::vector<float>* find(vasr_handle* h, const std::string& k) {
  auto it = h->staged.find(k);
  return it == h->staged.end() ? nullptr : &it->second;
}

int need(vasr_handle* h, const std::string& k, int64_t numel, const std::vector<float>** out) {
  const std::vector<float>* v = find(h, k);
  if (!v) return fail(VASR_ERR_STATE, "missing weight: " + k);
  if (numel >= 0 && (int64_t)v->size() != numel)
    return fail(VASR_ERR_SHAPE, "weight " + k + " has " + std::to_string(v->size()) + " elements, expected " +
                                    std::to_string(numel));
  *out = v;
  return VASR_OK;
}

template <typename T>
int upload(vasr_handle* h, const T* src, size_t n, T** dst) {
  void* p = nullptr;
  CK(cudaMalloc(&p, (n ? n : 1) * sizeof(T)));
  h->alloc_list->push_back(p);
  if (n) CK(cudaMemcpy(p, src, n * sizeof(T), cudaMemcpyHostToDevice));
  *dst = static_cast<T*>(p);
  return VASR_OK;
}

int up(vasr_handle* h, const std::string& k, int64_t numel, float** dst) {
  const std::vector<float>* v;
  RET(need(h, k, numel, &v));
  return upload(h, v->data(), v->size(), dst);
}

// FakeQuantize of a weight tensor, per output channel, symmetric int8, in the reference's operation order
// (quantize.py:99-133 with symmetric=True, per_channel=True, channel_dim=0; forward returns x + (dq - x)).
void fake_quant_rows(std::vector<float>& w, int64_t rows) {
  const int64_t cols = rows > 0 ? (int64_t)w.size() / rows : 0;
  for (int64_t r = 0; r < rows; ++r) {
    float* x = w.data() + r * cols;
    float lo = x[0], hi = x[0];
    for (int64_t c = 1; c < cols; ++c) { lo = fminf(lo, x[c]); hi = fmaxf(hi, x[c]); }
    float scale = fmaxf(fabsf(lo), fabsf(hi)) / 127.0f;
    if (scale < 1e-10f) scale = 1e-10f;
    for (int64_t c = 0; c < cols; ++c) {
      volatile float t = x[c] / scale;          // separately rounded, as eager PyTorch does
      float q = nearbyintf(t + 0.0f);
      q = fminf(fmaxf(q, -128.f), 127.f);
      volatile float dq = (q - 0.0f) * scale;
      volatile float diff = dq - x[c];
      x[c] = x[c] + diff;
    }
  }
}

// staged weight matrix `k` (rows x anything), fake-quantised when config 5 is on and the module is one of
// the 12 the reference replaces (every caller of this helper is)
int get_w(vasr_handle* h, const std::string& k, int64_t numel, int64_t rows, std::vector<float>* out) {
  const std::vector<float>* v;
  RET(need(h, k, numel, &v));
  *out = *v;
  if (h->quant) fake_quant_rows(*out, rows);
  return VASR_OK;
}
int up_w(vasr_handle* h, const std::string& k, int64_t numel, int64_t rows, float** dst) {
  std::vector<float> w;
  RET(get_w(h, k, numel, rows, &w));
  return upload(h, w.data(), w.size(), dst);
}

// y = Linear(LayerNorm(x)) = rstd * (x W'^T) - mean * rstd * s + b'   with   W' = W diag(gamma),
// b' = b + W beta,  s[n] = sum_k W'[n, k]:  the projection kernel takes x itself, its converter threads gather
// (mean, rstd) of the row they own and the epilogue applies the rest (GemmArgs::ln_s).  W: (N, K).
void fold_ln(const std::vector<float>& W, int64_t N, int64_t K, const float* bias, const float* gamma,
             const float* beta, std::vector<float>* Wf, std::vector<float>* bf, std::vector<float>* sf) {
  Wf->resize((size_t)N * K);
  bf->resize((size_t)N);
  sf->resize((size_t)N);
  for (int64_t n = 0; n < N; ++n) {
    double sb = bias ? (double)bias[n] : 0.0, ss = 0.0;
    for (int64_t k = 0; k < K; ++k) {
      const float w = W[(size_t)n * K + k];
      const float wf = w * gamma[k];
      (*Wf)[(size_t)n * K + k] = wf;
      sb += (double)w * (double)beta[k];
      ss += (double)wf;
    }
    (*bf)[(size_t)n] = (float)sb;
    (*sf)[(size_t)n] = (float)ss;
  }
}
// The folded form needs K = d in whole 32-deep k-blocks and more k-blocks than A slots (kernels.cuh, GemmArgs::ln_s);
// other widths keep the LayerNorm launch in front of the plain projection.
bool can_fold_ln(int d) { return d % 32 == 0 && d / 32 > 4; }
int upload_folded(vasr_handle* h, const std::vector<float>& W, int64_t N, int64_t K, const float* bias,
                  const std::string& gk, const std::string& bk, float** Wd, float** bd, float** sd) {
  const std::vector<float>*g, *b;
  RET(need(h, gk, K, &g));
  RET(need(h, bk, K, &b));
  std::vector<float> Wf, bf, sf;
  fold_ln(W, N, K, bias, g->data(), b->data(), &Wf, &bf, &sf);
  RET(upload(h, Wf.data(), Wf.size(), Wd));
  RET(upload(h, bf.data(), bf.size(), bd));
  return upload(h, sf.data(), sf.size(), sd);
}

// Row r' of the permuted fusion projection (3 C rows: gate | local | global stacked): the 192-column tile t holds,
// for its two 32-channel halves a, the chunks gate | local | global of channels 64 t + 32 a .. + 31, so that one
// epilogue warp (three chunks) has everything the mix of its 32 channels needs.
int gate_perm_row(int rp, int C) {
  const int t = rp / 192, a = (rp % 192) / 96, j = (rp % 96) / 32, i = rp % 32;
  return j * C + 64 * t + 32 * a + i;
}

int pack_block(vasr_handle* h, const std::string& p, int N, int expand, int ks, BlockW* w) {
  const int d = h->cfg.d_model, di = d * expand;
  w->N = N;
  w->di = di;
  w->ks = ks;
  RET(up(h, p + "norm1.weight", d, &w->ln1_g));
  RET(up(h, p + "norm1.bias", d, &w->ln1_b));
  RET(up(h, p + "norm2.weight", d, &w->ln2_g));
  RET(up(h, p + "norm2.bias", d, &w->ln2_b));
  RET(up(h, p + "conv.weight", (int64_t)d * ks, &w->conv_w));
  RET(up(h, p + "conv.bias", d, &w->conv_b));
  const std::vector<float>*alog, *xw, *dw, *db;
  RET(need(h, p + "ssm.A_log", N, &alog));
  std::vector<float> A(N);
  int structured = 1;
  for (int n = 0; n < N; ++n) {
    A[n] = -expf((*alog)[n]);
    if (fabsf((*alog)[n] - logf((float)(n + 1))) > 1e-6f) structured = 0;
  }
  w->structured = structured;
  RET(upload(h, A.data(), A.size(), &w->A));
  RET(up(h, p + "ssm.D", di, &w->D));
  RET(up(h, p + "ssm.in_proj.weight", (int64_t)2 * di * d, &w->w_in));
  RET(need(h, p + "ssm.x_proj.weight", (int64_t)2 * N * di, &xw));
  RET(need(h, p + "ssm.dt_proj.weight", (int64_t)di * di, &dw));
  RET(need(h, p + "ssm.dt_proj.bias", di, &db));
  std::vector<float> wx((size_t)(2 * N + di) * di), bx((size_t)2 * N + di, 0.f);
  memcpy(wx.data(), xw->data(), xw->size() * sizeof(float));
  memcpy(wx.data() + xw->size(), dw->data(), dw->size() * sizeof(float));
  memcpy(bx.data() + 2 * N, db->data(), db->size() * sizeof(float));
  RET(upload(h, wx.data(), wx.size(), &w->w_xdt));
  RET(upload(h, bx.data(), bx.size(), &w->b_xdt));
  RET(up(h, p + "ssm.out_proj.weight", (int64_t)d * di, &w->w_out));
  const std::vector<float>*f1w, *f1b;
  RET(need(h, p + "ffn.0.weight", (int64_t)di * d, &f1w));
  RET(need(h, p + "ffn.0.bias", di, &f1b));
  w->s_f1 = nullptr;
  // ffn.0's folded variant exists for the 192-column tiling only: di = 192 a + (0 or >= 128) columns
  if (can_fold_ln(d) && (di % 192 == 0 || di % 192 >= 128)) {
    RET(upload_folded(h, *f1w, di, d, f1b->data(), p + "norm2.weight", p + "norm2.bias", &w->w_f1, &w->b_f1, &w->s_f1));
  } else {
    RET(upload(h, f1w->data(), f1w->size(), &w->w_f1));
    RET(upload(h, f1b->data(), f1b->size(), &w->b_f1));
  }
  RET(up(h, p + "ffn.3.weight", (int64_t)d * di, &w->w_f2));
  RET(up(h, p + "ffn.3.bias", d, &w->b_f2));
  return VASR_OK;
}

// default front-end tables (float32 restatement of audio.py:97, 164-199)
void default_window(std::vector<float>& w) {
  w.resize(N_FFT);
  for (int i = 0; i < N_FFT; ++i) w[i] = (float)(0.5 - 0.5 * cos(2.0 * M_PI * i / N_FFT));
}
void default_filterbank(int n_mels, std::vector<float>& fb) {
  fb.assign((size_t)n_mels * N_FREQ, 0.f);
  auto lin = [](float a, float b, int steps, int i) {
    float step = (b - a) / (float)(steps - 1);
    return i < steps / 2 ? a + step * (float)i : b - step * (float)(steps - 1 - i);
  };
  const float mel_max = 2595.f * log10f(1.f + 8000.f / 700.f);
  std::vector<float> hz(n_mels + 2);
  for (int i = 0; i < n_mels + 2; ++i) hz[i] = 700.f * (powf(10.f, lin(0.f, mel_max, n_mels + 2, i) / 2595.f) - 1.f);
  for (int j = 0; j < n_mels; ++j)
    for (int k = 0; k < N_FREQ; ++k) {
      const float f = lin(0.f, 8000.f, N_FREQ, k);
      const float up_ = (f - hz[j]) / (hz[j + 1] - hz[j] + 1e-10f);
      const float dn = (hz[j + 2] - f) / (hz[j + 2] - hz[j + 1] + 1e-10f);
      const float v = up_ < dn ? up_ : dn;
      fb[(size_t)j * N_FREQ + k] = v > 0.f ? v : 0.f;
    }
}

int pack_frontend_impl(vasr_handle* h);
int setup_qsites(vasr_handle* h);
void free_splits(vasr_handle* h);
int pack_frontend(vasr_handle* h) {
  CK(cudaDeviceSynchronize());
  free_splits(h);
  for (void* p : h->frontend_allocs) cudaFree(p);
  h->frontend_allocs.clear();
  h->alloc_list = &h->frontend_allocs;
  const int r = pack_frontend_impl(h);
  h->alloc_list = &h->weight_allocs;
  return r;
}
int pack_frontend_impl(vasr_handle* h) {
  const int n_mels = h->cfg.mel_bins;
  std::vector<float> win, fb;
  if (const std::vector<float>* v = find(h, "frontend.window")) {
    if ((int)v->size() != N_FFT) return fail(VASR_ERR_SHAPE, "frontend.window must have 400 elements");
    win = *v;
  } else {
    default_window(win);
  }
  if (const std::vector<float>* v = find(h, "frontend.mel_filterbank")) {
    if ((int64_t)v->size() != (int64_t)n_mels * N_FREQ)
      return fail(VASR_ERR_SHAPE, "frontend.mel_filterbank must be n_mels x 201");
    fb = *v;
  } else {
    default_filterbank(n_mels, fb);
  }
  RET(upload(h, win.data(), win.size(), &h->win));
  std::vector<float> tw((size_t)2 * N_FFT);
  for (int m = 0; m < N_FFT; ++m) {
    const double ang = 2.0 * M_PI * (double)m / (double)N_FFT;
    tw[2 * m] = (float)cos(ang);
    tw[2 * m + 1] = (float)(-sin(ang));
  }
  RET(upload(h, tw.data(), tw.size(), &h->tw400));
  std::vector<int> lo(n_mels), off(n_mels + 1, 0);
  std::vector<float> wts;
  for (int j = 0; j < n_mels; ++j) {
    int a = -1, b = -1;
    for (int k = 0; k < N_FREQ; ++k)
      if (fb[(size_t)j * N_FREQ + k] != 0.f) {
        if (a < 0) a = k;
        b = k;
      }
    lo[j] = a < 0 ? 0 : a;
    if (a >= 0)
      for (int k = a; k <= b; ++k) wts.push_back(fb[(size_t)j * N_FREQ + k]);
    off[j + 1] = (int)wts.size();
  }
  RET(upload(h, lo.data(), lo.size(), &h->fb_lo));
  RET(upload(h, off.data(), off.size(), &h->fb_off));
  RET(upload(h, wts.data(), wts.size(), &h->fb_w));
  return VASR_OK;
}

void free_splits(vasr_handle* h) {
  for (auto& kv : h->w_split) cudaFree(kv.second);
  h->w_split.clear();
}

void free_weights(vasr_handle* h) {
  free_splits(h);
  for (void* p : h->weight_allocs) cudaFree(p);
  h->weight_allocs.clear();
  h->local.clear();
  h->global.clear();
  h->committed = false;
}

// ---------------------------------------------------------------- launch sequences ------
#define KL(expr)                                                                            \
  do {                                                                                      \
    cudaError_t e_ = (expr);                                                                \
    if (e_ != cudaSuccess)                                                                  \
      return fail(e_ == cudaErrorInvalidValue ? VASR_ERR_UNSUPPORTED : VASR_ERR_CUDA,       \
                  std::string(#expr) + ": " + cudaGetErrorString(e_));                      \
  } while (0)

// one projection.  Every projection of the model runs on the tensor-core kernel whatever its row
// count, so a row's result does not depend on how many utterances share the batch (the sharding
// rule of DESIGN.md section 5); the CUDA-core kernel serves the DFT rows and unaligned views.
// [W_hi | W_lo] for the tensor-core kernel: made on the device the first time a weight matrix is used
// (warm-up), then reused until the weights are re-committed.
int split_of(vasr_handle* h, const float* W, int64_t numel, cudaStream_t s, const float** out) {
  auto it = h->w_split.find(W);
  if (it == h->w_split.end()) {
    void* p = nullptr;
    CK(cudaMalloc(&p, (size_t)2 * numel * sizeof(float)));
    KL(launch_split_tf32(W, static_cast<float*>(p), numel, s));
    it = h->w_split.emplace(W, static_cast<float*>(p)).first;
  }
  *out = it->second;
  return VASR_OK;
}

int gemm(vasr_handle* h, GemmArgs& g, cudaStream_t s);
// Calibration of the output FakeQuantize nodes of one projection: the reference's FakeQuantize in training
// mode takes min / max of the tensor it is about to quantise (quantize.py:86-88, 99-121), i.e. of the module's
// own fp32 output given already-quantised inputs.  Probe = the same projection without quantisation,
// activation, positional encoding or residual, into scratch; then min / max per module and the new scales.
int calibrate_site(vasr_handle* h, const GemmArgs& g, const QSite& q, float* scratch, cudaStream_t s) {
  GemmArgs p = g;
  p.C = scratch; p.ldc = g.N;
  p.q_scale = p.q_zp = nullptr;
  p.act = ACT_NONE; p.act_from = 0;
  p.resid = nullptr; p.pe_time = p.pe_freq = nullptr;
  RET(gemm(h, p, s));
  for (int i = 0; i < q.nmod; ++i) {
    KL(launch_minmax(scratch, g.N, g.M, q.c0[i], q.nc[i], h->q_mm, s, &h->launches));
    KL(launch_set_qparams(h->q_mm, q.qs, q.qz, q.c0[i], q.nc[i], s, &h->launches));
  }
  return VASR_OK;
}

int gemm_impl(vasr_handle* h, GemmArgs& g, cudaStream_t s);
int gemm(vasr_handle* h, GemmArgs& g, cudaStream_t s) {
  if (!h->prof) return gemm_impl(h, g, s);
  vasr_handle::ProfEntry pe;
  pe.tag = "M" + std::to_string(g.M) + " K" + std::to_string(g.K) + " N" + std::to_string(g.N) + " act" +
           std::to_string(g.act) + (g.resid ? " resid" : "") + (g.pe_time ? " pe" : "") + (g.q_scale ? " quant" : "");
  CK(cudaEventCreate(&pe.e0));
  CK(cudaEventCreate(&pe.e1));
  CK(cudaEventRecord(pe.e0, s));
  const int r = gemm_impl(h, g, s);
  CK(cudaEventRecord(pe.e1, s));
  h->prof_ev.push_back(pe);
  return r;
}

// Every projection of the model runs on the tcgen05 kernel; a view it cannot take (alignment, tensor-map limits)
// is an error, never a silent change of kernel.
int gemm_impl(vasr_handle* h, GemmArgs& g, cudaStream_t s) {
  RET(split_of(h, g.W, g.N * g.K, s, &g.W_split));
  const cudaError_t e = launch_gemm_tc(g, h->num_sms, s, &h->launches);
  if (e == cudaErrorNotSupported) {
    (void)cudaGetLastError();
    return fail(VASR_ERR_UNSUPPORTED, "projection " + std::to_string(g.M) + " x " + std::to_string(g.K) + " -> " +
                                          std::to_string(g.N) + ": view not supported by the tensor-core kernel "
                                          "(16-byte alignment of rows, K % 4, N % 4)");
  }
  if (e != cudaSuccess) return fail(VASR_ERR_CUDA, std::string("launch_gemm_tc: ") + cudaGetErrorString(e));
  ++h->tc_launches;
  return VASR_OK;
}

// site >= 0: the projection hosts quantised modules (only meaningful while quant_active)
int gemm_q(vasr_handle* h, GemmArgs& g, int site, float* qscratch, cudaStream_t s) {
  if (site >= 0 && h->quant_active) {
    const QSite& q = h->qsite[site];
    g.q_scale = q.qs;
    g.q_zp = q.qz;
    if (h->calibrating) RET(calibrate_site(h, g, q, qscratch, s));
  }
  return gemm(h, g, s);
}

int linear(vasr_handle* h, const float* A, int64_t lda, const float* W, const float* bias, float* C, int64_t ldc,
           int64_t M, int64_t K, int64_t N, int act, int act_from, const float* resid, int64_t ldr,
           cudaStream_t s, int site = -1, float* qscratch = nullptr) {
  GemmArgs g;
  g.A = A; g.lda = lda; g.W = W; g.bias = bias; g.C = C; g.ldc = ldc;
  g.M = M; g.N = N; g.K = K; g.act = act; g.act_from = act_from; g.resid = resid; g.ldr = ldr;
  return gemm_q(h, g, site, qscratch, s);
}
// Linear(LayerNorm(A rows)) with the LayerNorm folded into the projection (fold_ln): W, bias, colsum are the folded set
int linear_ln(vasr_handle* h, const Work& k, const float* A, int64_t lda, const float* W, const float* bias,
              const float* colsum, float* C, int64_t ldc, int64_t M, int64_t K, int64_t N, int act, cudaStream_t s) {
  GemmArgs g;
  g.A = A; g.lda = lda; g.W = W; g.bias = bias; g.C = C; g.ldc = ldc;
  g.M = M; g.N = N; g.K = K; g.act = act; g.act_from = 0;
  g.ln_s = colsum; g.ln_stats = k.lnstat;
  return gemm(h, g, s);
}


int run_scan(vasr_handle* h, const BlockW& w, const Work& k, int64_t B, int64_t L, int quirk, cudaStream_t s) {
  const int di = w.di;
  const int64_t ld = 2 * w.N + di;
  ScanArgs a;
  a.x = k.xz; a.ldx = 2 * di;
  a.z = k.xz + di; a.ldz = 2 * di;
  a.Bm = k.bcdt; a.ldb = ld;
  a.Cm = k.bcdt + w.N; a.ldc = ld;
  a.dt = k.bcdt + 2 * w.N; a.lddt = ld;
  a.A = w.A; a.D = w.D;
  a.y = k.yg; a.ldy = di;
  a.B = B; a.L = L; a.Di = di; a.N = w.N;
  a.parallel_quirk = quirk;
  a.structured_a = w.structured;
  a.num_sms = h->num_sms;
  const bool t = h->timing && h->ev_used + 2 <= (int)h->ev.size();
  if (t) cudaEventRecord(h->ev[h->ev_used], s);
  KL(launch_selective_scan(a, s, &h->launches));
  if (t) {
    cudaEventRecord(h->ev[h->ev_used + 1], s);
    h->ev_used += 2;
  }
  return VASR_OK;
}

// SSMBlock._forward_impl (ssm.py:404-427): x (M, d) in k.xa -> result in k.xa; xb/u/xz/... scratch
int run_block(vasr_handle* h, const BlockW& w, const Work& k, float* x, float* x1, int64_t B, int64_t L, int quirk,
              cudaStream_t s) {
  const int d = h->cfg.d_model, di = w.di;
  const int64_t M = B * L;
  KL(launch_ln_dwconv(x, k.u, w.ln1_g, w.ln1_b, w.conv_w, w.conv_b, B, L, d, w.ks, s, &h->launches));
  RET(linear(h, k.u, d, w.w_in, nullptr, k.xz, 2 * di, M, d, 2 * di, ACT_NONE, 0, nullptr, 0, s));
  RET(linear(h, k.xz, 2 * di, w.w_xdt, w.b_xdt, k.bcdt, 2 * w.N + di, M, di, 2 * w.N + di, ACT_SOFTPLUS, 2 * w.N,
             nullptr, 0, s));
  RET(run_scan(h, w, k, B, L, quirk, s));
  RET(linear(h, k.yg, di, w.w_out, nullptr, x1, d, M, di, d, ACT_NONE, 0, x, d, s));
  if (w.s_f1) {
    RET(linear_ln(h, k, x1, d, w.w_f1, w.b_f1, w.s_f1, k.hbuf, di, M, d, di, ACT_GELU, s));    // norm2 folded into ffn.0
  } else {
    KL(launch_layer_norm(x1, d, k.u, d, w.ln2_g, w.ln2_b, M, d, s, &h->launches));
    RET(linear(h, k.u, d, w.w_f1, w.b_f1, k.hbuf, di, M, d, di, ACT_GELU, 0, nullptr, 0, s));
  }
  RET(linear(h, k.hbuf, di, w.w_f2, w.b_f2, x, d, M, di, d, ACT_NONE, 0, x1, d, s));
  return VASR_OK;
}

int quirk_for(const vasr_handle* h, int stack, int scan_mode) {
  if (scan_mode < 0) scan_mode = stack == 0 ? h->cfg.scan_mode : VASR_SCAN_PARALLEL;
  return scan_mode == VASR_SCAN_PARALLEL ? 1 : 0;
}

// HierarchicalGlobalContext.forward on local features already in k.cat[:, :d] -> k.fused
int run_global_context(vasr_handle* h, const Dims& q, const Work& k, cudaStream_t s) {
  const int d = q.d, att = q.att;
  KL(launch_adaptive_pool(k.cat, 2 * d, k.gb, q.B, q.L, q.K1, d, s, &h->launches, k.rag, RAG_L, RAG_K1));
  RET(linear(h, k.gb, d, h->p1_w, h->p1_b, k.ga, d, q.Mg, d, d, ACT_NONE, 0, nullptr, 0, s, Q_P1, k.qscratch));
  for (size_t i = 0; i < h->global.size(); ++i)
    RET(run_block(h, h->global[i], k, k.ga, k.gb, q.B, q.K1, quirk_for(h, 1, -1), s));
  KL(launch_layer_norm(k.ga, d, k.ga, d, h->glo_g, h->glo_b, q.Mg, d, s, &h->launches));
  KL(launch_adaptive_pool(k.ga, d, k.g2, q.B, q.K1, q.K2, d, s, &h->launches, k.rag, RAG_K1, RAG_K2));
  RET(linear(h, k.g2, d, h->p2_w, h->p2_b, k.g2n, d, q.M2, d, d, ACT_NONE, 0, nullptr, 0, s, Q_P2, k.qscratch));
  if (h->w_kv_ln) {          // fp32 model: norm1 / norm2 folded into the k | v and q projections
    RET(linear_ln(h, k, k.g2n, d, h->w_kv_ln, h->b_kv_ln, h->s_kv, k.kv, 2 * att, q.M2, d, 2 * att, ACT_NONE, s));
    RET(linear_ln(h, k, k.cat, 2 * d, h->w_q_ln, h->b_q_ln, h->s_q, k.qb, att, q.M, d, att, ACT_NONE, s));
  } else {
    KL(launch_layer_norm(k.g2n, d, k.g2n, d, h->n1_g, h->n1_b, q.M2, d, s, &h->launches));
    RET(linear(h, k.g2n, d, h->w_kv, h->b_kv, k.kv, 2 * att, q.M2, d, 2 * att, ACT_NONE, 0, nullptr, 0, s, Q_KV, k.qscratch));
    KL(launch_layer_norm(k.cat, 2 * d, k.u, d, h->n2_g, h->n2_b, q.M, d, s, &h->launches));
    RET(linear(h, k.u, d, h->w_q, h->b_q, k.qb, att, q.M, d, att, ACT_NONE, 0, nullptr, 0, s, Q_Q, k.qscratch));
  }
  KL(launch_attention(k.qb, att, k.kv, k.ob, att, q.B, q.L, q.K2, h->cfg.attention_heads,
                      att / h->cfg.attention_heads, s, &h->launches, k.rag));
  RET(linear(h, k.ob, att, h->w_o, h->b_o, k.cat + d, 2 * d, q.M, att, d, ACT_NONE, 0, nullptr, 0, s, Q_O, k.qscratch));
  if (h->w_f3p) {            // fp32 model: gate | local | global in one projection whose epilogue mixes them
    GemmArgs g;
    g.A = k.cat; g.lda = 2 * d; g.W = h->w_f3p; g.bias = h->b_f3p; g.C = k.fm; g.ldc = d;
    g.M = q.M; g.N = 3 * d; g.K = 2 * d; g.gate = 1;
    RET(gemm(h, g, s));
  } else {
    RET(linear(h, k.cat, 2 * d, h->w_f3, h->b_f3, k.f3, 3 * d, q.M, 2 * d, 3 * d, ACT_NONE, 0, nullptr, 0, s, Q_F3, k.qscratch));
    KL(launch_gate_mix(k.f3, k.fm, q.M, d, s, &h->launches));
  }
  RET(linear(h, k.fm, d, h->w_fo, h->b_fo, k.fused, d, q.M, d, d, ACT_NONE, 0, nullptr, 0, s, Q_FO, k.qscratch));
  return VASR_OK;
}

// logits == NULL (fp32 model only): greedy decode, the head leaves per-frame argmax partials in k.amax_* instead
int run_ctc_head(vasr_handle* h, const Dims& q, const Work& k, const float* x, float* logits, cudaStream_t s) {
  if (h->w_ctc_ln) {         // fp32 model: the head's LayerNorm folded into its projection
    GemmArgs g;
    g.A = x; g.lda = q.d; g.W = h->w_ctc_ln; g.bias = h->b_ctc_ln; g.C = logits; g.ldc = q.V;
    g.M = q.M; g.N = q.V; g.K = q.d;
    g.ln_s = h->s_ctc; g.ln_stats = k.lnstat;
    if (!logits) { g.amax_val = k.amax_val; g.amax_idx = k.amax_idx; }
    return gemm(h, g, s);
  }
  if (!logits) return fail(VASR_ERR_STATE, "the FakeQuantize model decodes from its logits");
  KL(launch_layer_norm(x, q.d, k.u, q.d, h->ctc_g, h->ctc_b, q.M, q.d, s, &h->launches));
  RET(linear(h, k.u, q.d, h->w_ctc, h->b_ctc, logits, q.V, q.M, q.d, q.V, ACT_NONE, 0, nullptr, 0, s, Q_CTC, k.qscratch));
  return VASR_OK;
}

// padded mel (k.melpad) -> logits
int run_model(vasr_handle* h, const Dims& q, const Work& k, float* logits, float* f_tb, float* f_local,
              float* f_fused, cudaStream_t s) {
  const int d = q.d;
  if (q.L > h->pe_rows)
    return fail(VASR_ERR_SHAPE, "sequence of " + std::to_string(q.L) + " tokens exceeds the positional table (" +
                                    std::to_string(h->pe_rows) + " rows, model.py:87,125)");
  GemmArgs g;
  g.A = k.melpad; g.lda = 2 * q.n_mels; g.rows_per_batch = q.L; g.batch_stride = q.Tp * q.n_mels;
  g.W = h->tb_w; g.bias = h->tb_b; g.C = k.xa; g.ldc = d;
  g.M = q.M; g.N = d; g.K = 3 * q.n_mels;
  g.act = ACT_GELU; g.act_from = 0;
  g.pe_time = h->pe_time; g.pe_freq = h->pe_freq; g.pe_half = d / 2; g.pe_rows = q.L;
  RET(gemm_q(h, g, Q_TB, k.qscratch, s));
  KL(launch_layer_norm(k.xa, d, k.xa, d, h->tb_g, h->tb_bt, q.M, d, s, &h->launches));
  if (f_tb) CK(cudaMemcpyAsync(f_tb, k.xa, (size_t)q.M * d * sizeof(float), cudaMemcpyDeviceToDevice, s));
  for (size_t i = 0; i < h->local.size(); ++i)
    RET(run_block(h, h->local[i], k, k.xa, k.xb, q.B, q.L, quirk_for(h, 0, -1), s));
  KL(launch_layer_norm(k.xa, d, k.cat, 2 * d, h->loc_g, h->loc_b, q.M, d, s, &h->launches));
  if (f_local)
    CK(cudaMemcpy2DAsync(f_local, (size_t)d * sizeof(float), k.cat, (size_t)2 * d * sizeof(float),
                         (size_t)d * sizeof(float), (size_t)q.M, cudaMemcpyDeviceToDevice, s));
  RET(run_global_context(h, q, k, s));
  if (f_fused) CK(cudaMemcpyAsync(f_fused, k.fused, (size_t)q.M * d * sizeof(float), cudaMemcpyDeviceToDevice, s));
  RET(run_ctc_head(h, q, k, k.fused, logits, s));
  return VASR_OK;
}

// PCM (device) -> k.raw (+ the partial statistics launch_mel_finish merges, when normalize)
int run_mel(vasr_handle* h, const Dims& q, const Work& k, const float* pcm, int normalize, cudaStream_t s) {
  KL(launch_mel_fft(pcm, k.raw, normalize ? k.part : nullptr, q.B, q.S, q.T, q.n_mels, h->fb_lo, h->fb_off, h->fb_w,
                    h->win, h->tw400, s, &h->launches, k.rag));
  return VASR_OK;
}

// Host PCM -> k.raw (+ partial statistics): HOST_SLICES transfers on copy_stream, each followed on `s` by the
// log-mel of its utterances; then the statistics of the whole batch.
int run_mel_from_host(vasr_handle* h, const Dims& q, const Work& k, const float* pcm_host, cudaStream_t s) {
  const int64_t per = (q.B + vasr_handle::HOST_SLICES - 1) / vasr_handle::HOST_SLICES;
  const int64_t nblk = mel_fft_blocks(q.T);
  CK(cudaEventRecord(h->copy_gate, s));                        // the stage buffer is free once `s` got here
  CK(cudaStreamWaitEvent(h->copy_stream, h->copy_gate, 0));
  int i = 0;
  for (int64_t b0 = 0; b0 < q.B; b0 += per, ++i) {
    const int64_t nb = q.B - b0 < per ? q.B - b0 : per;
    CK(cudaMemcpyAsync(k.pcm_stage + b0 * q.S, pcm_host + b0 * q.S, (size_t)nb * q.S * sizeof(float),
                       cudaMemcpyHostToDevice, h->copy_stream));
    CK(cudaEventRecord(h->slice_ev[i], h->copy_stream));
    CK(cudaStreamWaitEvent(s, h->slice_ev[i], 0));
    KL(launch_mel_fft(k.pcm_stage + b0 * q.S, k.raw + b0 * q.T * q.n_mels, k.part + b0 * nblk * q.n_mels * 2, nb, q.S,
                      q.T, q.n_mels, h->fb_lo, h->fb_off, h->fb_w, h->win, h->tw400, s, &h->launches,
                      k.rag ? k.rag + b0 * RAG_STRIDE : nullptr));
  }
  return VASR_OK;
}

int check_ready(const vasr_handle* h) {
  if (!h) return fail(VASR_ERR_INVALID, "null handle");
  if (!h->committed) return fail(VASR_ERR_STATE, "weights not committed (call vasr_commit_weights)");
  return VASR_OK;
}

// Binds the handle's device for the duration of one entry point and puts the caller's device back afterwards
// (a model on cuda:1 must not move a single-process multi-GPU program's current device).
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess || prev == dev) prev = -1;
    cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// Orders one workspace-using call after the previous one on the same handle (see vasr_handle::call_done).
struct CallOrder {
  vasr_handle* h;
  cudaStream_t s;
  CallOrder(vasr_handle* h_, cudaStream_t s_) : h(h_), s(s_) {
    if (h->call_pending && h->call_stream != s) cudaStreamWaitEvent(s, h->call_done, 0);
  }
  ~CallOrder() {
    if (cudaEventRecord(h->call_done, s) == cudaSuccess) {
      h->call_stream = s;
      h->call_pending = true;
    }
  }
  CallOrder(const CallOrder&) = delete;
  CallOrder& operator=(const CallOrder&) = delete;
};

void timing_begin(vasr_handle* h, cudaStream_t s) {
  h->ev_used = 0;
  h->ev_total = false;
  if (h->timing) {
    cudaEventRecord(h->ev_t0, s);
    h->ev_total = true;
  }
}
void timing_end(vasr_handle* h, cudaStream_t s) {
  if (h->timing) cudaEventRecord(h->ev_t1, s);
}

// the nine projections that host the twelve quantised modules, with their column ranges
int setup_qsites(vasr_handle* h) {
  const int d = h->cfg.d_model, att = h->cfg.attention_dim, V = h->cfg.vocab_size;
  auto site = [&](int id, int N, std::initializer_list<const char*> names, std::initializer_list<int> widths) {
    QSite& q = h->qsite[id];
    q.N = N;
    q.nmod = 0;
    int c = 0;
    auto w = widths.begin();
    for (const char* nm : names) {
      q.name[q.nmod] = nm; q.c0[q.nmod] = c; q.nc[q.nmod] = *w;
      c += *w; ++w; ++q.nmod;
    }
  };
  site(Q_TB, d, {"temporal_binding.conv"}, {d});
  site(Q_P1, d, {"global_context.pool1.pool_proj"}, {d});
  site(Q_P2, d, {"global_context.pool2.pool_proj"}, {d});
  site(Q_Q, att, {"global_context.cross_attention.q_proj"}, {att});
  site(Q_KV, 2 * att, {"global_context.cross_attention.k_proj", "global_context.cross_attention.v_proj"}, {att, att});
  site(Q_O, d, {"global_context.cross_attention.out_proj"}, {d});
  site(Q_F3, 3 * d, {"global_context.fusion.gate_proj.0", "global_context.fusion.local_proj",
                     "global_context.fusion.global_proj"}, {d, d, d});
  site(Q_FO, d, {"global_context.fusion.out_proj"}, {d});
  site(Q_CTC, V, {"ctc_head.proj.2"}, {V});
  for (int i = 0; i < Q_SITES; ++i) {
    QSite& q = h->qsite[i];
    std::vector<float> zeros((size_t)q.N, 0.f);     // scale 0 = pass-through until calibrated (quantize.py:82-84)
    RET(upload(h, zeros.data(), zeros.size(), &q.qs));
    RET(upload(h, zeros.data(), zeros.size(), &q.qz));
  }
  if (!h->q_mm) {
    void* p = nullptr;
    CK(cudaMalloc(&p, 2 * sizeof(float)));
    h->q_mm = static_cast<float*>(p);
  }
  return VASR_OK;
}

QSite* find_module(vasr_handle* h, const char* module, int* idx) {
  for (int i = 0; i < Q_SITES; ++i)
    for (int j = 0; j < h->qsite[i].nmod; ++j)
      if (strcmp(h->qsite[i].name[j], module) == 0) {
        *idx = j;
        return &h->qsite[i];
      }
  return nullptr;
}

}  // namespace

// =========================================================================== C ABI =======
extern "C" {

const char* vasr_last_error(void) { return g_err.c_str(); }
const char* vasr_version(void) { return "libvasr 0.1 (sm_100a)"; }

int64_t vasr_num_frames(int64_t samples) { return 1 + samples / HOP; }
int64_t vasr_num_tokens(int64_t frames) { return (frames + 1) / 2; }

int vasr_create(const vasr_config* cfg, int device, vasr_handle** out) {
  if (!cfg || !out) return fail(VASR_ERR_INVALID, "null argument");
  *out = nullptr;
  const vasr_config& c = *cfg;
  if (c.scan_mode < 0 || c.scan_mode > 2) return fail(VASR_ERR_INVALID, "Unknown scan_mode");
  if (c.d_model <= 0 || c.d_model > 192 || (c.d_model % 16) != 0)
    return fail(VASR_ERR_UNSUPPORTED, "d_model must be a multiple of 16, at most 192");
  // the front end takes any width up to 128; the temporal-binding projection's constraint is checked at commit
  if (c.mel_bins < 1 || c.mel_bins > 128) return fail(VASR_ERR_UNSUPPORTED, "mel_bins must be in [1, 128]");
  auto n_ok = [](int n) { return n == 16 || n == 32 || n == 64; };
  if (!n_ok(c.ssm_state_dim) || !n_ok(c.global_ssm_state_dim))
    return fail(VASR_ERR_UNSUPPORTED, "ssm state_dim must be 16, 32 or 64");
  const int di = c.d_model * c.ssm_expand_ratio;
  if (c.ssm_expand_ratio < 1 || (di % 64) != 0 || (c.d_model * GLOBAL_EXPAND) % 64 != 0)
    return fail(VASR_ERR_UNSUPPORTED, "d_model*expand_ratio (and 2*d_model for the global stack) must be multiples of 64");
  if (c.ssm_kernel_size < 1 || c.ssm_kernel_size > 8) return fail(VASR_ERR_UNSUPPORTED, "ssm_kernel_size must be in [1, 8]");
  if (c.attention_heads < 1 || c.attention_dim % c.attention_heads != 0 || c.attention_dim / c.attention_heads > 16 ||
      c.attention_dim % 16 != 0 || c.attention_heads > 4)
    return fail(VASR_ERR_UNSUPPORTED, "attention_dim must be a multiple of 16 with head_dim <= 16 and at most 4 heads "
                                      "(the attention kernel runs 64 threads per head in a 256-thread CTA)");
  if (c.vocab_size < 1 || c.ssm_layers < 0 || c.global_ssm_layers < 0) return fail(VASR_ERR_INVALID, "bad sizes");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return fail(VASR_ERR_CUDA, "no CUDA device: libvasr has no CPU path");
  if (device < 0 || device >= ndev) return fail(VASR_ERR_INVALID, "bad device index");
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(VASR_ERR_CUDA, std::string("libvasr is built for sm_100a only; device is ") + prop.name);
  DeviceGuard dev_guard(device);
  vasr_handle* h = new vasr_handle();
  h->cfg = c;
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  h->prof = debug_env_int("VASR_PROF", 0);
  CK(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  for (auto& e : h->slice_ev) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->copy_gate, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->call_done, cudaEventDisableTiming));
  h->ev.resize(64);
  for (auto& e : h->ev) CK(cudaEventCreate(&e));
  CK(cudaEventCreate(&h->ev_t0));
  CK(cudaEventCreate(&h->ev_t1));
  RET(pack_frontend(h));
  *out = h;
  return VASR_OK;
}

void vasr_destroy(vasr_handle* h) {
  if (!h) return;
  DeviceGuard dev_guard(h->device);
  cudaDeviceSynchronize();
  free_weights(h);
  for (void* p : h->frontend_allocs) cudaFree(p);
  if (h->ws.base) cudaFree(h->ws.base);
  if (h->q_mm) cudaFree(h->q_mm);
  for (auto& e : h->ev) cudaEventDestroy(e);
  if (h->ev_t0) cudaEventDestroy(h->ev_t0);
  if (h->ev_t1) cudaEventDestroy(h->ev_t1);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  for (auto& e : h->slice_ev)
    if (e) cudaEventDestroy(e);
  if (h->copy_gate) cudaEventDestroy(h->copy_gate);
  if (h->call_done) cudaEventDestroy(h->call_done);
  for (int i = 0; i < vasr_handle::RAG_RING; ++i) {
    if (h->rag_pin[i]) cudaFreeHost(h->rag_pin[i]);
    if (h->rag_ev[i]) cudaEventDestroy(h->rag_ev[i]);
  }
  delete h;
}

int vasr_set_weight(vasr_handle* h, const char* name, const float* host, int64_t numel) {
  if (!h || !name || (!host && numel > 0) || numel < 0) return fail(VASR_ERR_INVALID, "null argument");
  const std::string k(name);
  static const char* prefixes[] = {"temporal_binding.", "local_ssm.", "global_context.", "ctc_head.", "frontend."};
  bool ok = false;
  for (const char* p : prefixes) ok = ok || k.rfind(p, 0) == 0;
  if (!ok) return fail(VASR_ERR_INVALID, "unknown weight name: " + k);
  h->staged[k].assign(host, host + numel);
  if (k.rfind("frontend.", 0) == 0) {  // front-end tables take effect at once, model weights at commit
    DeviceGuard dev_guard(h->device);
    return pack_frontend(h);
  }
  h->committed = false;
  return VASR_OK;
}

int vasr_commit_weights(vasr_handle* h) {
  if (!h) return fail(VASR_ERR_INVALID, "null handle");
  DeviceGuard dev_guard(h->device);
  CK(cudaDeviceSynchronize());
  free_weights(h);
  h->w_q_ln = h->b_q_ln = h->s_q = h->w_kv_ln = h->b_kv_ln = h->s_kv = nullptr;
  h->w_ctc_ln = h->b_ctc_ln = h->s_ctc = h->w_f3p = h->b_f3p = nullptr;
  const vasr_config& c = h->cfg;
  const int d = c.d_model, nm = c.mel_bins, att = c.attention_dim;
  if ((nm * 3) % 16 != 0)
    return fail(VASR_ERR_UNSUPPORTED, "mel_bins must make 3*mel_bins a multiple of 16 (the temporal-binding projection)");
  // temporal binding: conv.weight (d, mel, 3) -> (d, 3*mel) with k index = tap*mel + channel
  std::vector<float> cwv;
  RET(get_w(h, "temporal_binding.conv.weight", (int64_t)d * nm * 3, d, &cwv));
  const std::vector<float>* cw = &cwv;
  std::vector<float> tbw((size_t)d * 3 * nm);
  for (int o = 0; o < d; ++o)
    for (int ch = 0; ch < nm; ++ch)
      for (int j = 0; j < 3; ++j) tbw[(size_t)o * 3 * nm + j * nm + ch] = (*cw)[((size_t)o * nm + ch) * 3 + j];
  RET(upload(h, tbw.data(), tbw.size(), &h->tb_w));
  RET(up(h, "temporal_binding.conv.bias", d, &h->tb_b));
  const std::vector<float>* pt;
  RET(need(h, "temporal_binding.pos_encoding.pe_time", -1, &pt));
  if (pt->size() % (size_t)(d / 2) != 0) return fail(VASR_ERR_SHAPE, "pe_time must be (rows, d_model/2)");
  h->pe_rows = (int64_t)pt->size() / (d / 2);
  RET(upload(h, pt->data(), pt->size(), &h->pe_time));
  RET(up(h, "temporal_binding.pos_encoding.pe_freq", d - d / 2, &h->pe_freq));
  RET(up(h, "temporal_binding.norm.weight", d, &h->tb_g));
  RET(up(h, "temporal_binding.norm.bias", d, &h->tb_bt));
  h->local.resize(c.ssm_layers);
  for (int i = 0; i < c.ssm_layers; ++i)
    RET(pack_block(h, "local_ssm.layers." + std::to_string(i) + ".", c.ssm_state_dim, c.ssm_expand_ratio,
                   c.ssm_kernel_size, &h->local[i]));
  RET(up(h, "local_ssm.norm.weight", d, &h->loc_g));
  RET(up(h, "local_ssm.norm.bias", d, &h->loc_b));
  const std::string gc = "global_context.";
  h->global.resize(c.global_ssm_layers);
  for (int i = 0; i < c.global_ssm_layers; ++i)
    RET(pack_block(h, gc + "global_ssm.layers." + std::to_string(i) + ".", c.global_ssm_state_dim, GLOBAL_EXPAND,
                   GLOBAL_KS, &h->global[i]));
  RET(up(h, gc + "global_ssm.norm.weight", d, &h->glo_g));
  RET(up(h, gc + "global_ssm.norm.bias", d, &h->glo_b));
  RET(up_w(h, gc + "pool1.pool_proj.weight", (int64_t)d * d, d, &h->p1_w));
  RET(up(h, gc + "pool1.pool_proj.bias", d, &h->p1_b));
  RET(up_w(h, gc + "pool2.pool_proj.weight", (int64_t)d * d, d, &h->p2_w));
  RET(up(h, gc + "pool2.pool_proj.bias", d, &h->p2_b));
  RET(up(h, gc + "norm1.weight", d, &h->n1_g));
  RET(up(h, gc + "norm1.bias", d, &h->n1_b));
  RET(up(h, gc + "norm2.weight", d, &h->n2_g));
  RET(up(h, gc + "norm2.bias", d, &h->n2_b));
  RET(up_w(h, gc + "cross_attention.q_proj.weight", (int64_t)att * d, att, &h->w_q));
  RET(up(h, gc + "cross_attention.q_proj.bias", att, &h->b_q));
  const std::vector<float>*kb, *vb;
  std::vector<float> kwv, vwv;
  RET(get_w(h, gc + "cross_attention.k_proj.weight", (int64_t)att * d, att, &kwv));
  RET(need(h, gc + "cross_attention.k_proj.bias", att, &kb));
  RET(get_w(h, gc + "cross_attention.v_proj.weight", (int64_t)att * d, att, &vwv));
  RET(need(h, gc + "cross_attention.v_proj.bias", att, &vb));
  const std::vector<float>*kw = &kwv, *vw = &vwv;
  std::vector<float> wkv(*kw), bkv(*kb);
  wkv.insert(wkv.end(), vw->begin(), vw->end());
  bkv.insert(bkv.end(), vb->begin(), vb->end());
  RET(upload(h, wkv.data(), wkv.size(), &h->w_kv));
  RET(upload(h, bkv.data(), bkv.size(), &h->b_kv));
  if (!h->quant && can_fold_ln(d)) {
    const std::vector<float>*qw, *qb;
    RET(need(h, gc + "cross_attention.q_proj.weight", (int64_t)att * d, &qw));
    RET(need(h, gc + "cross_attention.q_proj.bias", att, &qb));
    RET(upload_folded(h, *qw, att, d, qb->data(), gc + "norm2.weight", gc + "norm2.bias", &h->w_q_ln, &h->b_q_ln, &h->s_q));
    RET(upload_folded(h, wkv, 2 * att, d, bkv.data(), gc + "norm1.weight", gc + "norm1.bias", &h->w_kv_ln, &h->b_kv_ln,
                      &h->s_kv));
  }
  RET(up_w(h, gc + "cross_attention.out_proj.weight", (int64_t)d * att, d, &h->w_o));
  RET(up(h, gc + "cross_attention.out_proj.bias", d, &h->b_o));
  // fusion: one (3d x 2d) projection of [local | ctx]: gate rows, then local_proj on the left
  // half, then global_proj on the right half (zeros elsewhere).
  const std::vector<float>*gb, *lb, *cb2;
  std::vector<float> gwv, lwv, cwv2;
  RET(get_w(h, gc + "fusion.gate_proj.0.weight", (int64_t)d * 2 * d, d, &gwv));
  RET(need(h, gc + "fusion.gate_proj.0.bias", d, &gb));
  RET(get_w(h, gc + "fusion.local_proj.weight", (int64_t)d * d, d, &lwv));
  RET(need(h, gc + "fusion.local_proj.bias", d, &lb));
  RET(get_w(h, gc + "fusion.global_proj.weight", (int64_t)d * d, d, &cwv2));
  RET(need(h, gc + "fusion.global_proj.bias", d, &cb2));
  const std::vector<float>*gw = &gwv, *lw = &lwv, *cw2 = &cwv2;
  std::vector<float> wf3((size_t)3 * d * 2 * d, 0.f), bf3;
  memcpy(wf3.data(), gw->data(), gw->size() * sizeof(float));
  for (int o = 0; o < d; ++o) {
    memcpy(&wf3[(size_t)(d + o) * 2 * d], &(*lw)[(size_t)o * d], d * sizeof(float));
    memcpy(&wf3[(size_t)(2 * d + o) * 2 * d + d], &(*cw2)[(size_t)o * d], d * sizeof(float));
  }
  bf3 = *gb;
  bf3.insert(bf3.end(), lb->begin(), lb->end());
  bf3.insert(bf3.end(), cb2->begin(), cb2->end());
  RET(upload(h, wf3.data(), wf3.size(), &h->w_f3));
  RET(upload(h, bf3.data(), bf3.size(), &h->b_f3));
  h->w_f3p = h->b_f3p = nullptr;
  if (!h->quant && d % 64 == 0) {
    std::vector<float> wp(wf3.size()), bp(bf3.size());
    for (int rp = 0; rp < 3 * d; ++rp) {
      const int r = gate_perm_row(rp, d);
      memcpy(&wp[(size_t)rp * 2 * d], &wf3[(size_t)r * 2 * d], (size_t)2 * d * sizeof(float));
      bp[(size_t)rp] = bf3[(size_t)r];
    }
    RET(upload(h, wp.data(), wp.size(), &h->w_f3p));
    RET(upload(h, bp.data(), bp.size(), &h->b_f3p));
  }
  RET(up_w(h, gc + "fusion.out_proj.weight", (int64_t)d * d, d, &h->w_fo));
  RET(up(h, gc + "fusion.out_proj.bias", d, &h->b_fo));
  RET(up(h, "ctc_head.proj.0.weight", d, &h->ctc_g));
  RET(up(h, "ctc_head.proj.0.bias", d, &h->ctc_b));
  RET(up_w(h, "ctc_head.proj.2.weight", (int64_t)c.vocab_size * d, c.vocab_size, &h->w_ctc));
  RET(up(h, "ctc_head.proj.2.bias", c.vocab_size, &h->b_ctc));
  if (!h->quant && can_fold_ln(d)) {
    const std::vector<float>*hw, *hb;
    RET(need(h, "ctc_head.proj.2.weight", (int64_t)c.vocab_size * d, &hw));
    RET(need(h, "ctc_head.proj.2.bias", c.vocab_size, &hb));
    RET(upload_folded(h, *hw, c.vocab_size, d, hb->data(), "ctc_head.proj.0.weight", "ctc_head.proj.0.bias", &h->w_ctc_ln,
                      &h->b_ctc_ln, &h->s_ctc));
  }
  h->quant_active = h->quant;
  if (h->quant_active) RET(setup_qsites(h));
  h->committed = true;
  return VASR_OK;
}

int vasr_log_mel(vasr_handle* h, const float* pcm_dev, int64_t B, int64_t S, int normalize, float* mel_dev,
                 void* stream) {
  if (!h) return fail(VASR_ERR_INVALID, "null handle");
  if (B < 0 || !pcm_dev || !mel_dev) return fail(VASR_ERR_INVALID, "null argument");
  if (S <= PAD) return fail(VASR_ERR_SHAPE, "reflect padding needs more than 200 samples (audio.py:100-101)");
  DeviceGuard dev_guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CallOrder call_order(h, s);
  const Dims q = make_dims(h, B, S, vasr_num_frames(S));
  Work k;
  RET(ensure_workspace(h, q, true, false, &k));
  RET(run_mel(h, q, k, pcm_dev, normalize, s));
  KL(launch_mel_finish(k.raw, mel_dev, q.B, q.T, q.n_mels, q.T, 0, s, &h->launches, nullptr,
                       normalize ? k.part : nullptr));
  return VASR_OK;
}

int vasr_forward(vasr_handle* h, const float* mel_dev, int64_t B, int64_t T, float* logits_dev, float* feat_tb_dev,
                 float* feat_local_dev, float* feat_fused_dev, void* stream) {
  RET(check_ready(h));
  if (B < 0 || T < 1 || !mel_dev || !logits_dev) return fail(VASR_ERR_INVALID, "null argument");
  DeviceGuard dev_guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CallOrder call_order(h, s);
  const Dims q = make_dims(h, B, 0, T);
  Work k;
  RET(ensure_workspace(h, q, false, false, &k));
  timing_begin(h, s);
  KL(launch_mel_finish(mel_dev, k.melpad, q.B, q.T, q.n_mels, q.Tp, 1, s, &h->launches));
  RET(run_model(h, q, k, logits_dev, feat_tb_dev, feat_local_dev, feat_fused_dev, s));
  timing_end(h, s);
  return VASR_OK;
}

int vasr_ssm_block(vasr_handle* h, int stack, int layer, int scan_mode, const float* x_dev, int64_t B, int64_t L,
                   float* out_dev, void* stream) {
  RET(check_ready(h));
  if (stack < 0 || stack > 1) return fail(VASR_ERR_INVALID, "stack must be 0 (local) or 1 (global)");
  const std::vector<BlockW>& blocks = stack == 0 ? h->local : h->global;
  if (layer < 0 || layer >= (int)blocks.size()) return fail(VASR_ERR_INVALID, "layer out of range");
  if (scan_mode > 2) return fail(VASR_ERR_INVALID, "Unknown scan_mode");
  DeviceGuard dev_guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CallOrder call_order(h, s);
  Dims q = make_dims(h, B, 0, 2 * L - 1);
  Work k;
  RET(ensure_workspace(h, q, false, false, &k));
  const size_t bytes = (size_t)B * L * q.d * sizeof(float);
  CK(cudaMemcpyAsync(k.xa, x_dev, bytes, cudaMemcpyDeviceToDevice, s));
  RET(run_block(h, blocks[layer], k, k.xa, k.xb, B, L, quirk_for(h, stack, scan_mode), s));
  CK(cudaMemcpyAsync(out_dev, k.xa, bytes, cudaMemcpyDeviceToDevice, s));
  return VASR_OK;
}

int vasr_global_context(vasr_handle* h, const float* local_dev, int64_t B, int64_t L, float* out_dev, void* stream) {
  RET(check_ready(h));
  DeviceGuard dev_guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CallOrder call_order(h, s);
  Dims q = make_dims(h, B, 0, 2 * L - 1);
  Work k;
  RET(ensure_workspace(h, q, false, false, &k));
  const size_t row = (size_t)q.d * sizeof(float);
  CK(cudaMemcpy2DAsync(k.cat, 2 * row, local_dev, row, row, (size_t)q.M, cudaMemcpyDeviceToDevice, s));
  RET(run_global_context(h, q, k, s));
  CK(cudaMemcpyAsync(out_dev, k.fused, (size_t)q.M * row, cudaMemcpyDeviceToDevice, s));
  return VASR_OK;
}

int vasr_ctc_head(vasr_handle* h, const float* x_dev, int64_t B, int64_t L, float* logits_dev, void* stream) {
  RET(check_ready(h));
  DeviceGuard dev_guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CallOrder call_order(h, s);
  Dims q = make_dims(h, B, 0, 2 * L - 1);
  Work k;
  RET(ensure_workspace(h, q, false, false, &k));
  RET(run_ctc_head(h, q, k, x_dev, logits_dev, s));
  return VASR_OK;
}

int vasr_selective_scan(const float* x, int64_t ldx, const float* dt, int64_t lddt, const float* A, const float* Bm,
                        int64_t ldb, const float* Cm, int64_t ldc, const float* D, const float* z, int64_t ldz,
                        float* y, int64_t ldy, int64_t B, int64_t L, int64_t Di, int64_t N, int scan_mode,
                        void* stream) {
  if (!x || !dt || !A || !Bm || !Cm || !y) return fail(VASR_ERR_INVALID, "null argument");
  if (scan_mode < 0 || scan_mode > 2) return fail(VASR_ERR_INVALID, "Unknown scan_mode");
  if (N != 16 && N != 32 && N != 64) return fail(VASR_ERR_UNSUPPORTED, "state_dim must be 16, 32 or 64");
  float ah[64];
  CK(cudaMemcpy(ah, A, (size_t)N * sizeof(float), cudaMemcpyDeviceToHost));
  int structured = 1;
  for (int n = 0; n < N; ++n)
    if (fabsf(ah[n] + (float)(n + 1)) > 2e-6f * (float)(n + 1)) structured = 0;
  ScanArgs a;
  a.x = x; a.ldx = ldx; a.dt = dt; a.lddt = lddt; a.z = z; a.ldz = ldz;
  a.Bm = Bm; a.ldb = ldb; a.Cm = Cm; a.ldc = ldc; a.A = A; a.D = D; a.y = y; a.ldy = ldy;
  a.B = B; a.L = L; a.Di = (int)Di; a.N = (int)N;
  a.parallel_quirk = scan_mode == VASR_SCAN_PARALLEL;
  a.structured_a = structured;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int dev = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&a.num_sms, cudaDevAttrMultiProcessorCount, dev));
  KL(launch_selective_scan(a, s, nullptr));
  return VASR_OK;
}

int vasr_ctc_greedy(const float* logits_dev, int64_t B, int64_t L, int64_t V, int blank, int collapse,
                    int32_t* tokens_dev, int32_t* lens_dev, void* stream) {
  if (!tokens_dev || !lens_dev || (!logits_dev && B * L > 0)) return fail(VASR_ERR_INVALID, "null argument");
  if (B <= 0) return VASR_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int32_t* pred = nullptr;
  CK(cudaMallocAsync(reinterpret_cast<void**>(&pred), (size_t)(B * L > 0 ? B * L : 1) * sizeof(int32_t), s));
  KL(launch_argmax(logits_dev, pred, B * L, (int)V, s, nullptr));
  KL(launch_ctc_collapse(pred, tokens_dev, lens_dev, B, L, blank, collapse, s, nullptr));
  CK(cudaFreeAsync(pred, s));
  return VASR_OK;
}

int vasr_ctc_greedy_timestamps(const float* logits_dev, int64_t B, int64_t L, int64_t V, int blank,
                               int32_t* tokens_dev, int32_t* starts_dev, int32_t* ends_dev, int32_t* lens_dev,
                               void* stream) {
  if (!tokens_dev || !starts_dev || !ends_dev || !lens_dev || (!logits_dev && B * L > 0))
    return fail(VASR_ERR_INVALID, "null argument");
  if (B <= 0) return VASR_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int32_t* pred = nullptr;
  CK(cudaMallocAsync(reinterpret_cast<void**>(&pred), (size_t)(B * L > 0 ? B * L : 1) * sizeof(int32_t), s));
  KL(launch_argmax(logits_dev, pred, B * L, (int)V, s, nullptr));
  KL(launch_ctc_runs(pred, tokens_dev, starts_dev, ends_dev, lens_dev, B, L, blank, s, nullptr));
  CK(cudaFreeAsync(pred, s));
  return VASR_OK;
}

struct vasr_lm {
  int device = 0, blank = 0;
  void* block = nullptr;   // every device table (lm.cu)
  LmView view;
  // a word LM: view is over word ids; the search's vocabulary size, the spelling trie and the word strings
  bool word = false;
  int64_t vocab = 0, lexicon = 0;
  void* lex_block = nullptr;
  LexView lex;
  std::unordered_map<std::string, int> word_id;
};

int vasr_lm_create_arpa(const char* path, const char* const* vocab, int64_t V, int blank, int device, vasr_lm** out) {
  if (!path || !vocab || !out) return fail(VASR_ERR_INVALID, "null argument");
  *out = nullptr;
  if (V < 1 || V >= 0x7fffffff) return fail(VASR_ERR_INVALID, "vocabulary size must be in [1, 2^31 - 1)");
  if (blank < 0 || blank >= V) return fail(VASR_ERR_INVALID, "blank token outside the vocabulary");
  LmHostTables t;
  std::string err;
  if (!lm_parse_arpa(path, vocab, (int)V, blank, &t, &err)) return fail(VASR_ERR_INVALID, err);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(VASR_ERR_CUDA, "no CUDA device: libvasr has no CPU path");
  if (device < 0) CK(cudaGetDevice(&device));
  if (device >= ndev) return fail(VASR_ERR_INVALID, "bad device index");
  DeviceGuard dev_guard(device);
  vasr_lm* lm = new vasr_lm;
  lm->device = device;
  lm->blank = blank;
  const cudaError_t e = lm_upload(t, &lm->block, &lm->view);
  if (e != cudaSuccess) {
    delete lm;
    return fail(VASR_ERR_CUDA, std::string("LM upload: ") + cudaGetErrorString(e));
  }
  *out = lm;
  return VASR_OK;
}

int vasr_lm_create_word_arpa(const char* path, const char* const* vocab, int64_t V, int blank, const char* delimiter,
                             int constrained, int device, vasr_lm** out) {
  if (!path || !vocab || !delimiter || !out) return fail(VASR_ERR_INVALID, "null argument");
  *out = nullptr;
  if (V < 1 || V >= 0x7fffffff) return fail(VASR_ERR_INVALID, "vocabulary size must be in [1, 2^31 - 1)");
  if (blank < 0 || blank >= V) return fail(VASR_ERR_INVALID, "blank token outside the vocabulary");
  LmHostTables t;
  LexHostTables x;
  std::string err;
  if (!lm_parse_word_arpa(path, vocab, (int)V, blank, delimiter, constrained != 0, &t, &x, &err))
    return fail(VASR_ERR_INVALID, err);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(VASR_ERR_CUDA, "no CUDA device: libvasr has no CPU path");
  if (device < 0) CK(cudaGetDevice(&device));
  if (device >= ndev) return fail(VASR_ERR_INVALID, "bad device index");
  DeviceGuard dev_guard(device);
  vasr_lm* lm = new vasr_lm;
  lm->device = device;
  lm->blank = blank;
  lm->word = true;
  lm->vocab = V;
  lm->lexicon = x.lexicon;
  for (size_t i = 0; i < x.words.size(); ++i) lm->word_id.emplace(x.words[i], (int)i);
  cudaError_t e = lm_upload(t, &lm->block, &lm->view);
  if (e == cudaSuccess) e = lex_upload(x, constrained != 0, &lm->lex_block, &lm->lex);
  if (e != cudaSuccess) {
    vasr_lm_destroy(lm);
    return fail(VASR_ERR_CUDA, std::string("LM upload: ") + cudaGetErrorString(e));
  }
  *out = lm;
  return VASR_OK;
}

void vasr_lm_destroy(vasr_lm* lm) {
  if (!lm) return;
  DeviceGuard dev_guard(lm->device);
  cudaFree(lm->block);
  cudaFree(lm->lex_block);
  delete lm;
}

int64_t vasr_lm_lexicon_size(const vasr_lm* lm) { return lm && lm->word ? lm->lexicon : -1; }

int vasr_lm_word_ids(const vasr_lm* lm, const char* const* words, int64_t n, int32_t* ids_host) {
  if (!lm || n < 0 || (n > 0 && (!words || !ids_host))) return fail(VASR_ERR_INVALID, "null argument");
  if (!lm->word) return fail(VASR_ERR_INVALID, "not a word LM");
  for (int64_t i = 0; i < n; ++i) {
    if (!words[i]) return fail(VASR_ERR_INVALID, "null word");
    auto it = lm->word_id.find(words[i]);
    if (it != lm->word_id.end()) ids_host[i] = it->second;
    else if (lm->lex.unk >= 0) ids_host[i] = lm->lex.unk;
    else return fail(VASR_ERR_INVALID, std::string("`") + words[i] + "` is not a word of the LM, which has no <unk>");
  }
  return VASR_OK;
}

int vasr_lm_order(const vasr_lm* lm) { return lm ? lm->view.order : 0; }

int vasr_lm_log_prob(const vasr_lm* lm, const int32_t* prefixes_dev, const int32_t* prefix_lens_dev, int64_t n,
                     const int32_t* tokens_dev, float* out_dev, void* stream) {
  if (!lm || n < 0) return fail(VASR_ERR_INVALID, "null argument");
  if (n == 0) return VASR_OK;
  if (!prefixes_dev || !prefix_lens_dev || !tokens_dev || !out_dev) return fail(VASR_ERR_INVALID, "null argument");
  DeviceGuard dev_guard(lm->device);
  KL(launch_lm_log_prob(lm->view, prefixes_dev, prefix_lens_dev, n, tokens_dev, out_dev,
                        static_cast<cudaStream_t>(stream)));
  return VASR_OK;
}

namespace {

// Argument checks shared by every search entry point (no device call): lm NULL runs the LM-free rule (lm_weight and
// word_score unused), a token LM the rule of beam_search_lm_kernel (word_score must be 0), a word LM that of
// beam_search_word_lm_kernel.  row_lens_host (optional): B frame counts, each in [0, L].
int beam_check(const int32_t* row_lens_host, int64_t B, int64_t L, int64_t V, int beam_width,
               int blank, const vasr_lm* lm, double lm_weight, double word_score, const int32_t* tokens_dev,
               const int32_t* lens_dev, const double* scores_dev) {
  if (!tokens_dev && B * beam_width * L > 0) return fail(VASR_ERR_INVALID, "null argument");
  if (!lens_dev || !scores_dev) return fail(VASR_ERR_INVALID, "null argument");
  if (beam_width < 1 || beam_width > 32) return fail(VASR_ERR_INVALID, "beam_width must be in [1, 32]");
  if (V < 1 || blank < 0 || blank >= V) return fail(VASR_ERR_INVALID, "blank token outside the vocabulary");
  if (lm) {
    const int64_t lv = lm->word ? lm->vocab : lm->view.V;
    if (V != lv)
      return fail(VASR_ERR_INVALID, "the LM is built for a vocabulary of " + std::to_string(lv) +
                                        " tokens, the logits have " + std::to_string(V));
    if (blank != lm->blank)
      return fail(VASR_ERR_INVALID, "the LM is built with blank token " + std::to_string(lm->blank) +
                                        ", the search uses " + std::to_string(blank));
    if (lm->word) {
      if (!std::isfinite(lm_weight) || lm_weight < 0)
        return fail(VASR_ERR_INVALID, "lm_weight must be finite and >= 0");
      if (!std::isfinite(word_score)) return fail(VASR_ERR_INVALID, "word_score must be finite");
    } else {
      if (!std::isfinite(lm_weight)) return fail(VASR_ERR_INVALID, "lm_weight must be finite");
      if (word_score != 0) return fail(VASR_ERR_INVALID, "word_score needs a word LM");
    }
  }
  if (row_lens_host)
    for (int64_t b = 0; b < B; ++b)
      if (row_lens_host[b] < 0 || row_lens_host[b] > L)
        return fail(VASR_ERR_SHAPE, "ragged search: every utterance needs between 0 and L frames (utterance " +
                                        std::to_string(b) + " has " + std::to_string(row_lens_host[b]) + ")");
  return VASR_OK;
}

// The body of every search entry point: checks, the device check, scratch sizing and the launches.  Frame counts
// come from the host (row_lens_host, uploaded here) or are already on the device (lens_dev at stride lens_stride:
// the RAG_L column of a fused call's ragged dims); neither: every utterance has L frames.
int beam_search(const float* logits_dev, const int32_t* row_lens_host, const int32_t* lens_dev, int lens_stride,
                int64_t B, int64_t L, int64_t V, int beam_width, int blank, const vasr_lm* lm, double lm_weight,
                double word_score, int32_t* tokens_dev, int32_t* out_lens_dev, double* scores_dev, cudaStream_t s) {
  if (!logits_dev && B * L > 0) return fail(VASR_ERR_INVALID, "null argument");
  RET(beam_check(row_lens_host, B, L, V, beam_width, blank, lm, lm_weight, word_score, tokens_dev, out_lens_dev,
                 scores_dev));
  if (B <= 0) return VASR_OK;
  int dev = 0;
  if (lm) {
    dev = lm->device;
    if (B * L > 0) {
      cudaPointerAttributes at = {};
      if (cudaPointerGetAttributes(&at, logits_dev) != cudaSuccess || at.type == cudaMemoryTypeUnregistered ||
          at.type == cudaMemoryTypeHost || at.device != lm->device) {
        cudaGetLastError();
        return fail(VASR_ERR_INVALID, "the logits are not device memory on the LM's device (" +
                                          std::to_string(lm->device) + ")");
      }
    }
  } else {
    CK(cudaGetDevice(&dev));
  }
  DeviceGuard dev_guard(dev);
  const int W = beam_width;
  // candidate tokens per frame (beam.cu says why these counts): LM-free W+1; word LM lexicon-free W+2; a token LM
  // and a constrained word LM list their own, so beam_rows gives them the log-softmax stats only
  int K = 0;
  if (!lm) K = (int)(V - 1 < W + 1 ? V - 1 : W + 1) > 0 ? (int)(V - 1 < W + 1 ? V - 1 : W + 1) : 1;
  else if (lm->word && !lm->lex.constrained) K = (int)(V - 1 < W + 2 ? (V - 1 > 0 ? V - 1 : 1) : W + 2);
  const int planes = !lm ? 3 : lm->word ? 9 : 5;
  const int64_t M = B * L, cap = 1 + L * W;
  float2* stats = nullptr;
  int32_t *top = nullptr, *trie = nullptr, *ulens = nullptr;
  float *trie_f = nullptr, *rows = nullptr;
  CK(cudaMallocAsync(reinterpret_cast<void**>(&stats), (size_t)(M > 0 ? M : 1) * sizeof(float2), s));
  if (K > 0) CK(cudaMallocAsync(reinterpret_cast<void**>(&top), (size_t)(M > 0 ? M : 1) * K * sizeof(int32_t), s));
  CK(cudaMallocAsync(reinterpret_cast<void**>(&trie), (size_t)planes * B * cap * sizeof(int32_t), s));
  if (lm) CK(cudaMallocAsync(reinterpret_cast<void**>(&trie_f), (size_t)B * cap * sizeof(float), s));
  if (lm && !lm->word) CK(cudaMallocAsync(reinterpret_cast<void**>(&rows), (size_t)B * W * V * sizeof(float), s));
  // The caller may reuse its array as soon as the call returns, and it may be pinned (then the copy would read it
  // whenever the stream gets there): copy it to pageable memory of our own first.  cudaMemcpyAsync stages a
  // pageable source before it returns, so this copy may go when the function does.
  std::vector<int32_t> row_lens;
  if (row_lens_host) {
    row_lens.assign(row_lens_host, row_lens_host + B);
    CK(cudaMallocAsync(reinterpret_cast<void**>(&ulens), (size_t)B * sizeof(int32_t), s));
    CK(cudaMemcpyAsync(ulens, row_lens.data(), (size_t)B * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    lens_dev = ulens;
    lens_stride = 1;
  }
  KL(launch_beam_rows(logits_dev, stats, top, M, (int)V, K, blank, L, lens_dev, lens_stride, s, nullptr));
  if (!lm)
    KL(launch_beam_search(logits_dev, stats, top, K, B, L, lens_dev, lens_stride, (int)V, W, blank, trie, cap,
                          tokens_dev, out_lens_dev, scores_dev, s, nullptr));
  else if (!lm->word)
    KL(launch_beam_search_lm(logits_dev, stats, lm->view, lm_weight, B, L, lens_dev, lens_stride, (int)V, W, blank,
                             trie, trie_f, cap, rows, tokens_dev, out_lens_dev, scores_dev, s));
  else
    KL(launch_beam_search_word_lm(logits_dev, stats, top, K, lm->view, lm->lex, lm_weight, word_score, B, L,
                                  lens_dev, lens_stride, (int)V, W, blank, trie, trie_f, cap, tokens_dev,
                                  out_lens_dev, scores_dev, s));
  CK(cudaFreeAsync(stats, s));
  if (top) CK(cudaFreeAsync(top, s));
  CK(cudaFreeAsync(trie, s));
  if (trie_f) CK(cudaFreeAsync(trie_f, s));
  if (rows) CK(cudaFreeAsync(rows, s));
  if (ulens) CK(cudaFreeAsync(ulens, s));
  return VASR_OK;
}

}  // namespace

int vasr_ctc_beam_search(const float* logits_dev, int64_t B, int64_t L, int64_t V, int beam_width, int blank,
                         int32_t* tokens_dev, int32_t* lens_dev, double* scores_dev, void* stream) {
  return beam_search(logits_dev, nullptr, nullptr, 0, B, L, V, beam_width, blank, nullptr, 0.0, 0.0, tokens_dev,
                     lens_dev, scores_dev, static_cast<cudaStream_t>(stream));
}

int vasr_ctc_beam_search_lm(const float* logits_dev, int64_t B, int64_t L, int64_t V, int beam_width, int blank,
                            const vasr_lm* lm, double lm_weight, int32_t* tokens_dev, int32_t* lens_dev,
                            double* scores_dev, void* stream) {
  if (!lm) return fail(VASR_ERR_INVALID, "null LM");
  if (lm->word) return fail(VASR_ERR_INVALID, "a word LM runs in vasr_ctc_beam_search_word_lm");
  return beam_search(logits_dev, nullptr, nullptr, 0, B, L, V, beam_width, blank, lm, lm_weight, 0.0, tokens_dev,
                     lens_dev, scores_dev, static_cast<cudaStream_t>(stream));
}

int vasr_ctc_beam_search_word_lm(const float* logits_dev, int64_t B, int64_t L, int64_t V, int beam_width, int blank,
                                 const vasr_lm* lm, double lm_weight, double word_score, int32_t* tokens_dev,
                                 int32_t* lens_dev, double* scores_dev, void* stream) {
  if (!lm) return fail(VASR_ERR_INVALID, "null LM");
  if (!lm->word) return fail(VASR_ERR_INVALID, "a token LM runs in vasr_ctc_beam_search_lm");
  return beam_search(logits_dev, nullptr, nullptr, 0, B, L, V, beam_width, blank, lm, lm_weight, word_score,
                     tokens_dev, lens_dev, scores_dev, static_cast<cudaStream_t>(stream));
}

int vasr_ctc_beam_search_ragged(const float* logits_dev, const int32_t* row_lens_host, int64_t B, int64_t L,
                                int64_t V, int beam_width, int blank, const vasr_lm* lm, double lm_weight,
                                double word_score, int32_t* tokens_dev, int32_t* lens_dev, double* scores_dev,
                                void* stream) {
  return beam_search(logits_dev, row_lens_host, nullptr, 0, B, L, V, beam_width, blank, lm, lm_weight, word_score,
                     tokens_dev, lens_dev, scores_dev, static_cast<cudaStream_t>(stream));
}

namespace {

// Argument checks of every alignment entry point (no device call).  Only the first target_lens[b] ids of a row are
// read.  row_lens_host (optional): B frame counts, each in [0, L].
int align_check(const int32_t* row_lens_host, int64_t B, int64_t L, int64_t V, int blank, const int32_t* targets_host,
                const int32_t* target_lens_host, int64_t U_max) {
  if (B < 0 || L < 0 || U_max < 0) return fail(VASR_ERR_SHAPE, "negative size");
  if (B > 0 && (!target_lens_host || (!targets_host && U_max > 0))) return fail(VASR_ERR_INVALID, "null argument");
  if (V < 1 || blank < 0 || blank >= V) return fail(VASR_ERR_INVALID, "blank token outside the vocabulary");
  for (int64_t b = 0; b < B; ++b) {
    const int64_t U = target_lens_host[b];
    if (U < 0 || U > U_max)
      return fail(VASR_ERR_SHAPE, "every target length must be in [0, U_max] (utterance " + std::to_string(b) +
                                      " has " + std::to_string(U) + ")");
    for (int64_t u = 0; u < U; ++u) {
      const int32_t id = targets_host[b * U_max + u];
      if (id < 0 || id >= V || id == blank)
        return fail(VASR_ERR_INVALID, "target id " + std::to_string(id) + " of utterance " + std::to_string(b) +
                                          " is outside the vocabulary or the blank");
    }
  }
  if (row_lens_host)
    for (int64_t b = 0; b < B; ++b)
      if (row_lens_host[b] < 0 || row_lens_host[b] > L)
        return fail(VASR_ERR_SHAPE, "ragged alignment: every utterance needs between 0 and L frames (utterance " +
                                        std::to_string(b) + " has " + std::to_string(row_lens_host[b]) + ")");
  return VASR_OK;
}

// The body of every alignment entry point after its checks: scratch, the row statistics and the alignment kernel.
// ll == NULL: Viterbi into labels / lps / scores; else the log-likelihood into ll.  Frame counts as beam_search.
int ctc_align_run(const float* logits_dev, const int32_t* row_lens_host, const int32_t* lens_dev, int lens_stride,
                  int64_t B, int64_t L, int64_t V, int blank, int log_probs, const int32_t* targets_host,
                  const int32_t* target_lens_host, int64_t U_max, int32_t* labels, float* lps, double* scores,
                  double* ll, cudaStream_t s) {
  if (B <= 0) return VASR_OK;
  const bool viterbi = ll == nullptr;
  int64_t U = 0;
  for (int64_t b = 0; b < B; ++b) U = target_lens_host[b] > U ? target_lens_host[b] : U;
  int threads = 0, E = 0;
  ctc_align_layout(U, viterbi, &threads, &E);
  int dev = 0, smem_max = 0;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const bool delta_smem = ctc_align_smem(threads, E, true) <= (size_t)smem_max;
  const int64_t M = B * L, words = ctc_align_words(U);
  // host arrays -> one pageable copy of our own ([target_lens | row_lens | targets]), so the caller may reuse its
  // arrays, pinned or not, as soon as the call returns (cudaMemcpyAsync stages a pageable source before returning)
  std::vector<int32_t> pack((size_t)(2 * B + B * U_max));
  std::copy(target_lens_host, target_lens_host + B, pack.begin());
  if (row_lens_host) std::copy(row_lens_host, row_lens_host + B, pack.begin() + B);
  if (U_max > 0) std::copy(targets_host, targets_host + B * U_max, pack.begin() + 2 * B);
  // scratch, released (stream-ordered) on every return, errors included
  struct Scratch {
    void* p[4] = {};
    cudaStream_t s;
    ~Scratch() {
      for (void* q : p)
        if (q) cudaFreeAsync(q, s);
    }
  } scratch{{}, s};
  CK(cudaMallocAsync(&scratch.p[0], pack.size() * sizeof(int32_t), s));
  int32_t* packed = static_cast<int32_t*>(scratch.p[0]);
  CK(cudaMemcpyAsync(packed, pack.data(), pack.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  if (row_lens_host) {
    lens_dev = packed + B;
    lens_stride = 1;
  }
  if (!log_probs) CK(cudaMallocAsync(&scratch.p[1], (size_t)(M > 0 ? M : 1) * sizeof(float2), s));
  if (!delta_smem) CK(cudaMallocAsync(&scratch.p[2], (size_t)B * E * threads * sizeof(double), s));
  if (viterbi) CK(cudaMallocAsync(&scratch.p[3], (size_t)(M > 0 ? M : 1) * words * sizeof(uint32_t), s));
  float2* stats = static_cast<float2*>(scratch.p[1]);
  if (!log_probs) KL(launch_beam_rows(logits_dev, stats, nullptr, M, (int)V, 0, blank, L, lens_dev, lens_stride, s,
                                      nullptr));
  KL(launch_ctc_align(logits_dev, stats, B, L, (int)V, blank, lens_dev, lens_stride, packed + 2 * B, U_max, packed,
                      threads, E, static_cast<double*>(scratch.p[2]), static_cast<uint32_t*>(scratch.p[3]), words,
                      labels, lps, viterbi ? scores : ll, s));
  return VASR_OK;
}

int ctc_align_entry(const float* logits_dev, const int32_t* row_lens_host, int64_t B, int64_t L, int64_t V, int blank,
                    int log_probs, const int32_t* targets_host, const int32_t* target_lens_host, int64_t U_max,
                    int32_t* labels, float* lps, double* scores, double* ll, void* stream) {
  if (!logits_dev && B * L > 0) return fail(VASR_ERR_INVALID, "null argument");
  RET(align_check(row_lens_host, B, L, V, blank, targets_host, target_lens_host, U_max));
  return ctc_align_run(logits_dev, row_lens_host, nullptr, 0, B, L, V, blank, log_probs, targets_host,
                       target_lens_host, U_max, labels, lps, scores, ll, static_cast<cudaStream_t>(stream));
}

}  // namespace

int vasr_ctc_align(const float* logits_dev, const int32_t* row_lens_host, int64_t B, int64_t L, int64_t V, int blank,
                   int log_probs, const int32_t* targets_host, const int32_t* target_lens_host, int64_t U_max,
                   int32_t* frame_labels_dev, float* frame_log_probs_dev, double* scores_dev, void* stream) {
  if (!scores_dev || ((!frame_labels_dev || !frame_log_probs_dev) && B * L > 0))
    return fail(VASR_ERR_INVALID, "null argument");
  return ctc_align_entry(logits_dev, row_lens_host, B, L, V, blank, log_probs, targets_host, target_lens_host, U_max,
                         frame_labels_dev, frame_log_probs_dev, scores_dev, nullptr, stream);
}

int vasr_ctc_log_likelihood(const float* logits_dev, const int32_t* row_lens_host, int64_t B, int64_t L, int64_t V,
                            int blank, int log_probs, const int32_t* targets_host, const int32_t* target_lens_host,
                            int64_t U_max, double* ll_dev, void* stream) {
  if (!ll_dev) return fail(VASR_ERR_INVALID, "null argument");
  return ctc_align_entry(logits_dev, row_lens_host, B, L, V, blank, log_probs, targets_host, target_lens_host, U_max,
                         nullptr, nullptr, nullptr, ll_dev, stream);
}

// Per-utterance dims of a ragged batch -> k.ragbuf, k.rag.  `lens` (host) are samples (from_samples) or mel
// frames; each utterance gets the dims make_dims would give it alone.
static int upload_ragged(vasr_handle* h, const Dims& q, Work& k, const int32_t* lens, bool from_samples,
                         cudaStream_t s) {
  const int64_t count = q.B * RAG_STRIDE;
  if (count > h->rag_pin_cap) {
    CK(cudaDeviceSynchronize());
    for (int i = 0; i < vasr_handle::RAG_RING; ++i) {
      if (h->rag_pin[i]) CK(cudaFreeHost(h->rag_pin[i]));
      h->rag_pin[i] = nullptr;
      CK(cudaHostAlloc(reinterpret_cast<void**>(&h->rag_pin[i]), (size_t)count * sizeof(int32_t), cudaHostAllocDefault));
      if (!h->rag_ev[i]) CK(cudaEventCreateWithFlags(&h->rag_ev[i], cudaEventDisableTiming));
    }
    h->rag_pin_cap = count;
  }
  const int slot = h->rag_next;
  h->rag_next = (slot + 1) % vasr_handle::RAG_RING;
  CK(cudaEventSynchronize(h->rag_ev[slot]));      // the upload that last used this slot has been consumed
  int32_t* host = h->rag_pin[slot];
  for (int64_t i = 0; i < count; ++i) host[i] = 0;
  for (int64_t b = 0; b < q.B; ++b) {
    const int64_t n = lens[b];
    if (from_samples) {
      if (n <= PAD || n > q.S)
        return fail(VASR_ERR_SHAPE, "ragged batch: every utterance needs more than 200 and at most S samples");
    } else if (n < 1 || n > q.T) {
      return fail(VASR_ERR_SHAPE, "ragged batch: every utterance needs between 1 and T frames");
    }
    const Dims u = make_dims(h, 1, from_samples ? n : 0, from_samples ? vasr_num_frames(n) : n);
    int32_t* r = host + b * RAG_STRIDE;
    r[RAG_S] = (int32_t)(from_samples ? n : 0);
    r[RAG_T] = (int32_t)u.T;
    r[RAG_L] = (int32_t)u.L;
    r[RAG_K1] = (int32_t)u.K1;
    r[RAG_K2] = (int32_t)u.K2;
  }
  CK(cudaMemcpyAsync(k.ragbuf, host, (size_t)count * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  CK(cudaEventRecord(h->rag_ev[slot], s));
  k.rag = k.ragbuf;
  return VASR_OK;
}

static int transcribe_impl(vasr_handle* h, const float* pcm_dev, const float* pcm_host, int64_t B, int64_t S,
                           int32_t* tokens_dev, int32_t* lens_dev, int32_t* tokens_host, int32_t* lens_host,
                           cudaStream_t s, const int32_t* sample_lens = nullptr) {
  const bool host = pcm_host != nullptr;
  CallOrder call_order(h, s);
  const Dims q = make_dims(h, B, S, vasr_num_frames(S));
  Work k;
  const bool from_parts = h->w_ctc_ln != nullptr;       // fp32 model: the head's epilogue does the argmax, no logits
  RET(ensure_workspace(h, q, true, !from_parts, &k, host));
  if (sample_lens) RET(upload_ragged(h, q, k, sample_lens, true, s));
  if (host) {
    tokens_dev = k.tok_stage;
    lens_dev = k.len_stage;
  }
  timing_begin(h, s);
  if (host) RET(run_mel_from_host(h, q, k, pcm_host, s));
  else RET(run_mel(h, q, k, pcm_dev, 1, s));
  KL(launch_mel_finish(k.raw, k.melpad, q.B, q.T, q.n_mels, q.Tp, 1, s, &h->launches, k.rag, k.part));
  RET(run_model(h, q, k, from_parts ? nullptr : k.logits, nullptr, nullptr, nullptr, s));
  if (from_parts) {
    KL(launch_ctc_collapse(k.pred, tokens_dev, lens_dev, q.B, q.L, 0, 1, s, &h->launches, k.rag, k.amax_val, k.amax_idx,
                           argmax_slots(q.V)));
  } else {
    KL(launch_argmax(k.logits, k.pred, q.M, q.V, s, &h->launches));
    KL(launch_ctc_collapse(k.pred, tokens_dev, lens_dev, q.B, q.L, 0, 1, s, &h->launches, k.rag));
  }
  timing_end(h, s);
  if (host) {
    CK(cudaMemcpyAsync(tokens_host, tokens_dev, (size_t)q.M * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(lens_host, lens_dev, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  return VASR_OK;
}

int vasr_transcribe(vasr_handle* h, const float* pcm_dev, int64_t B, int64_t S, int32_t* tokens_dev,
                    int32_t* lens_dev, void* stream) {
  RET(check_ready(h));
  if (B < 0 || !pcm_dev || !tokens_dev || !lens_dev) return fail(VASR_ERR_INVALID, "null argument");
  if (S <= PAD) return fail(VASR_ERR_SHAPE, "reflect padding needs more than 200 samples (audio.py:100-101)");
  DeviceGuard dev_guard(h->device);
  return transcribe_impl(h, pcm_dev, nullptr, B, S, tokens_dev, lens_dev, nullptr, nullptr,
                         static_cast<cudaStream_t>(stream));
}

int vasr_transcribe_host(vasr_handle* h, const float* pcm_host, int64_t B, int64_t S, int32_t* tokens_host,
                         int32_t* lens_host) {
  RET(check_ready(h));
  if (B <= 0 || !pcm_host || !tokens_host || !lens_host) return fail(VASR_ERR_INVALID, "null argument");
  if (S <= PAD) return fail(VASR_ERR_SHAPE, "reflect padding needs more than 200 samples (audio.py:100-101)");
  DeviceGuard dev_guard(h->device);
  return transcribe_impl(h, nullptr, pcm_host, B, S, nullptr, nullptr, tokens_host, lens_host, h->own_stream);
}

int vasr_transcribe_ragged(vasr_handle* h, const float* pcm_dev, const int32_t* sample_lens_host, int64_t B,
                           int64_t S, int32_t* tokens_dev, int32_t* lens_dev, void* stream) {
  RET(check_ready(h));
  if (B < 0 || !pcm_dev || !tokens_dev || !lens_dev || !sample_lens_host)
    return fail(VASR_ERR_INVALID, "null argument");
  if (S <= PAD) return fail(VASR_ERR_SHAPE, "reflect padding needs more than 200 samples (audio.py:100-101)");
  DeviceGuard dev_guard(h->device);
  return transcribe_impl(h, pcm_dev, nullptr, B, S, tokens_dev, lens_dev, nullptr, nullptr,
                         static_cast<cudaStream_t>(stream), sample_lens_host);
}

int vasr_transcribe_ragged_host(vasr_handle* h, const float* pcm_host, const int32_t* sample_lens_host, int64_t B,
                                int64_t S, int32_t* tokens_host, int32_t* lens_host) {
  RET(check_ready(h));
  if (B <= 0 || !pcm_host || !tokens_host || !lens_host || !sample_lens_host)
    return fail(VASR_ERR_INVALID, "null argument");
  if (S <= PAD) return fail(VASR_ERR_SHAPE, "reflect padding needs more than 200 samples (audio.py:100-101)");
  DeviceGuard dev_guard(h->device);
  return transcribe_impl(h, nullptr, pcm_host, B, S, nullptr, nullptr, tokens_host, lens_host, h->own_stream,
                         sample_lens_host);
}

// PCM -> n-best: transcribe_impl's sequence with the logits-writing CTC head (vasr_forward's, for the fp32 and the
// FakeQuantize model alike) and the prefix beam search in place of the greedy decode.  A ragged batch's search
// reads each utterance's token count from the uploaded dims (RAG_L).  Host variant: results come back through
// device scratch and the call synchronises once at the end.
static int transcribe_beam_impl(vasr_handle* h, const float* pcm_dev, const float* pcm_host,
                                const int32_t* sample_lens, int64_t B, int64_t S, int beam_width, const vasr_lm* lm,
                                double lm_weight, double word_score, int32_t* tokens, int32_t* lens, double* scores,
                                cudaStream_t s) {
  const bool host = pcm_host != nullptr;
  if (lm && lm->device != h->device)
    return fail(VASR_ERR_INVALID, "the LM is on device " + std::to_string(lm->device) + ", the model on " +
                                      std::to_string(h->device));
  const Dims q = make_dims(h, B, S, vasr_num_frames(S));
  // every argument of the search is checked before any device work (sample_lens by upload_ragged below)
  RET(beam_check(nullptr, B, q.L, q.V, beam_width, 0, lm, lm_weight, word_score, tokens, lens, scores));
  if (B == 0) return VASR_OK;
  CallOrder call_order(h, s);
  Work k;
  RET(ensure_workspace(h, q, true, true, &k, host));
  if (sample_lens) RET(upload_ragged(h, q, k, sample_lens, true, s));
  const int64_t W = beam_width;
  int32_t *tok_dev = tokens, *len_dev = lens;
  double* sc_dev = scores;
  // host variant: device copies of the results, released (stream-ordered) on every return, errors included
  struct Stage {
    void* p[3] = {};
    cudaStream_t s;
    ~Stage() {
      for (void* q : p)
        if (q) cudaFreeAsync(q, s);
    }
  } stage{{}, s};
  if (host) {
    CK(cudaMallocAsync(&stage.p[0], (size_t)B * W * q.L * sizeof(int32_t), s));
    CK(cudaMallocAsync(&stage.p[1], (size_t)B * W * sizeof(int32_t), s));
    CK(cudaMallocAsync(&stage.p[2], (size_t)B * W * sizeof(double), s));
    tok_dev = static_cast<int32_t*>(stage.p[0]);
    len_dev = static_cast<int32_t*>(stage.p[1]);
    sc_dev = static_cast<double*>(stage.p[2]);
  }
  timing_begin(h, s);
  if (host) RET(run_mel_from_host(h, q, k, pcm_host, s));
  else RET(run_mel(h, q, k, pcm_dev, 1, s));
  KL(launch_mel_finish(k.raw, k.melpad, q.B, q.T, q.n_mels, q.Tp, 1, s, &h->launches, k.rag, k.part));
  RET(run_model(h, q, k, k.logits, nullptr, nullptr, nullptr, s));
  RET(beam_search(k.logits, nullptr, k.rag ? k.rag + RAG_L : nullptr, RAG_STRIDE, q.B, q.L, q.V, beam_width, 0, lm,
                  lm_weight, word_score, tok_dev, len_dev, sc_dev, s));
  timing_end(h, s);
  if (host) {
    CK(cudaMemcpyAsync(tokens, tok_dev, (size_t)B * W * q.L * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(lens, len_dev, (size_t)B * W * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(scores, sc_dev, (size_t)B * W * sizeof(double), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
  }
  return VASR_OK;
}

int vasr_transcribe_beam(vasr_handle* h, const float* pcm_dev, const int32_t* sample_lens_host, int64_t B, int64_t S,
                         int beam_width, const vasr_lm* lm, double lm_weight, double word_score, int32_t* tokens_dev,
                         int32_t* lens_dev, double* scores_dev, void* stream) {
  RET(check_ready(h));
  if (B < 0 || !pcm_dev) return fail(VASR_ERR_INVALID, "null argument");
  if (S <= PAD) return fail(VASR_ERR_SHAPE, "reflect padding needs more than 200 samples (audio.py:100-101)");
  DeviceGuard dev_guard(h->device);
  return transcribe_beam_impl(h, pcm_dev, nullptr, sample_lens_host, B, S, beam_width, lm, lm_weight, word_score,
                              tokens_dev, lens_dev, scores_dev, static_cast<cudaStream_t>(stream));
}

int vasr_transcribe_beam_host(vasr_handle* h, const float* pcm_host, const int32_t* sample_lens_host, int64_t B,
                              int64_t S, int beam_width, const vasr_lm* lm, double lm_weight, double word_score,
                              int32_t* tokens_host, int32_t* lens_host, double* scores_host) {
  RET(check_ready(h));
  if (B <= 0 || !pcm_host) return fail(VASR_ERR_INVALID, "null argument");
  if (S <= PAD) return fail(VASR_ERR_SHAPE, "reflect padding needs more than 200 samples (audio.py:100-101)");
  DeviceGuard dev_guard(h->device);
  return transcribe_beam_impl(h, nullptr, pcm_host, sample_lens_host, B, S, beam_width, lm, lm_weight, word_score,
                              tokens_host, lens_host, scores_host, h->own_stream);
}

// PCM -> forced alignment: transcribe_beam_impl's sequence (log-mel, model, the logits-writing CTC head, blank 0, a
// ragged batch's token counts from RAG_L) with the Viterbi alignment in place of the search.
int vasr_align(vasr_handle* h, const float* pcm_dev, const int32_t* sample_lens_host, int64_t B, int64_t S,
               const int32_t* targets_host, const int32_t* target_lens_host, int64_t U_max, int32_t* frame_labels_dev,
               float* frame_log_probs_dev, double* scores_dev, void* stream) {
  RET(check_ready(h));
  if (B < 0 || !pcm_dev || !frame_labels_dev || !frame_log_probs_dev || !scores_dev)
    return fail(VASR_ERR_INVALID, "null argument");
  if (S <= PAD) return fail(VASR_ERR_SHAPE, "reflect padding needs more than 200 samples (audio.py:100-101)");
  const Dims q = make_dims(h, B, S, vasr_num_frames(S));
  // every argument of the alignment is checked before any device work (sample_lens by upload_ragged below)
  RET(align_check(nullptr, B, q.L, q.V, 0, targets_host, target_lens_host, U_max));
  if (B == 0) return VASR_OK;
  DeviceGuard dev_guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CallOrder call_order(h, s);
  Work k;
  RET(ensure_workspace(h, q, true, true, &k, false));
  if (sample_lens_host) RET(upload_ragged(h, q, k, sample_lens_host, true, s));
  timing_begin(h, s);
  RET(run_mel(h, q, k, pcm_dev, 1, s));
  KL(launch_mel_finish(k.raw, k.melpad, q.B, q.T, q.n_mels, q.Tp, 1, s, &h->launches, k.rag, k.part));
  RET(run_model(h, q, k, k.logits, nullptr, nullptr, nullptr, s));
  RET(ctc_align_run(k.logits, nullptr, k.rag ? k.rag + RAG_L : nullptr, RAG_STRIDE, q.B, q.L, q.V, 0, 0, targets_host,
                    target_lens_host, U_max, frame_labels_dev, frame_log_probs_dev, scores_dev, nullptr, s));
  timing_end(h, s);
  return VASR_OK;
}

int vasr_forward_ragged(vasr_handle* h, const float* mel_dev, const int32_t* frame_lens_host, int64_t B, int64_t T,
                        float* logits_dev, void* stream) {
  RET(check_ready(h));
  if (B < 0 || T < 1 || !mel_dev || !logits_dev || !frame_lens_host) return fail(VASR_ERR_INVALID, "null argument");
  DeviceGuard dev_guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CallOrder call_order(h, s);
  const Dims q = make_dims(h, B, 0, T);
  Work k;
  RET(ensure_workspace(h, q, false, false, &k));
  RET(upload_ragged(h, q, k, frame_lens_host, false, s));
  timing_begin(h, s);
  KL(launch_mel_finish(mel_dev, k.melpad, q.B, q.T, q.n_mels, q.Tp, 1, s, &h->launches, k.rag));
  RET(run_model(h, q, k, logits_dev, nullptr, nullptr, nullptr, s));
  timing_end(h, s);
  return VASR_OK;
}

int vasr_linear(const float* x_dev, int64_t ldx, const float* w_dev, const float* bias_dev, float* out_dev,
                int64_t ldo, int64_t M, int64_t K, int64_t N, int act, void* stream) {
  if (!x_dev || !w_dev || !out_dev) return fail(VASR_ERR_INVALID, "null argument");
  if (act < 0 || act > 3) return fail(VASR_ERR_INVALID, "unknown activation");
  GemmArgs g;
  g.A = x_dev; g.lda = ldx; g.W = w_dev; g.bias = bias_dev; g.C = out_dev; g.ldc = ldo;
  g.M = M; g.N = N; g.K = K; g.act = act; g.act_from = 0;
  KL(launch_gemm(g, static_cast<cudaStream_t>(stream), nullptr));
  return VASR_OK;
}

int vasr_set_quantization(vasr_handle* h, int enabled) {
  if (!h) return fail(VASR_ERR_INVALID, "null handle");
  if ((enabled != 0) != (h->quant != 0)) {
    h->quant = enabled != 0;
    h->committed = false;      // weights are re-packed (fake-quantised or not) at the next commit
  }
  return VASR_OK;
}

int vasr_calibrate(vasr_handle* h, const float* mel_dev, int64_t B, int64_t T, void* stream) {
  RET(check_ready(h));
  if (!h->quant_active) return fail(VASR_ERR_STATE, "quantisation is not enabled (vasr_set_quantization + commit)");
  if (B <= 0 || T < 1 || !mel_dev) return fail(VASR_ERR_INVALID, "null argument");
  DeviceGuard dev_guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CallOrder call_order(h, s);
  const Dims q = make_dims(h, B, 0, T);
  Work k;
  RET(ensure_workspace(h, q, false, true, &k));
  KL(launch_mel_finish(mel_dev, k.melpad, q.B, q.T, q.n_mels, q.Tp, 1, s, &h->launches));
  h->calibrating = 1;
  const int r = run_model(h, q, k, k.logits, nullptr, nullptr, nullptr, s);
  h->calibrating = 0;
  return r;
}

int vasr_get_quant_params(vasr_handle* h, const char* module, float* scale, float* zero_point) {
  if (!h || !module || !scale || !zero_point) return fail(VASR_ERR_INVALID, "null argument");
  if (!h->quant_active) return fail(VASR_ERR_STATE, "quantisation is not enabled");
  int j = 0;
  QSite* q = find_module(h, module, &j);
  if (!q) return fail(VASR_ERR_INVALID, std::string("not a quantised module: ") + module);
  DeviceGuard dev_guard(h->device);
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(scale, q->qs + q->c0[j], sizeof(float), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(zero_point, q->qz + q->c0[j], sizeof(float), cudaMemcpyDeviceToHost));
  return VASR_OK;
}

int vasr_set_quant_params(vasr_handle* h, const char* module, float scale, float zero_point) {
  if (!h || !module) return fail(VASR_ERR_INVALID, "null argument");
  if (!h->quant_active) return fail(VASR_ERR_STATE, "quantisation is not enabled");
  int j = 0;
  QSite* q = find_module(h, module, &j);
  if (!q) return fail(VASR_ERR_INVALID, std::string("not a quantised module: ") + module);
  DeviceGuard dev_guard(h->device);
  CK(cudaDeviceSynchronize());
  std::vector<float> sv((size_t)q->nc[j], scale), zv((size_t)q->nc[j], zero_point);
  CK(cudaMemcpy(q->qs + q->c0[j], sv.data(), sv.size() * sizeof(float), cudaMemcpyHostToDevice));
  CK(cudaMemcpy(q->qz + q->c0[j], zv.data(), zv.size() * sizeof(float), cudaMemcpyHostToDevice));
  return VASR_OK;
}

int vasr_quant_site(vasr_handle* h, const char* module, const float* x_dev, int64_t B, int64_t R, float* out_dev,
                    int32_t* n_out, int32_t* col0, int32_t* ncol, void* stream) {
  RET(check_ready(h));
  if (!module) return fail(VASR_ERR_INVALID, "null argument");
  if (!h->quant_active) return fail(VASR_ERR_STATE, "quantisation is not enabled (vasr_set_quantization + commit)");
  int j = 0;
  QSite* q = find_module(h, module, &j);
  if (!q) return fail(VASR_ERR_INVALID, std::string("not a quantised module: ") + module);
  const int site = (int)(q - h->qsite);
  if (n_out) *n_out = q->N;
  if (col0) *col0 = q->c0[j];
  if (ncol) *ncol = q->nc[j];
  if (!x_dev || !out_dev) return B * R > 0 ? fail(VASR_ERR_INVALID, "null argument") : VASR_OK;
  if (B <= 0 || R <= 0) return VASR_OK;
  DeviceGuard dev_guard(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  CallOrder call_order(h, s);
  const int d = h->cfg.d_model, att = h->cfg.attention_dim;
  GemmArgs g;
  g.act = ACT_NONE;
  g.C = out_dev; g.ldc = q->N; g.N = q->N;
  if (site == Q_TB) {
    const Dims dm = make_dims(h, B, 0, R);
    Work k;
    RET(ensure_workspace(h, dm, false, false, &k));
    KL(launch_mel_finish(x_dev, k.melpad, dm.B, dm.T, dm.n_mels, dm.Tp, 1, s, &h->launches));
    g.A = k.melpad; g.lda = 2 * dm.n_mels; g.rows_per_batch = dm.L; g.batch_stride = dm.Tp * dm.n_mels;
    g.W = h->tb_w; g.bias = h->tb_b; g.M = dm.M; g.K = 3 * dm.n_mels;
  } else {
    struct { const float* w; const float* b; int K; } tab[Q_SITES] = {
        {nullptr, nullptr, 0}, {h->p1_w, h->p1_b, d}, {h->p2_w, h->p2_b, d}, {h->w_q, h->b_q, d},
        {h->w_kv, h->b_kv, d}, {h->w_o, h->b_o, att}, {h->w_f3, h->b_f3, 2 * d}, {h->w_fo, h->b_fo, d},
        {h->w_ctc, h->b_ctc, d}};
    g.A = x_dev; g.lda = tab[site].K; g.W = tab[site].w; g.bias = tab[site].b; g.M = B * R; g.K = tab[site].K;
  }
  g.q_scale = q->qs;
  g.q_zp = q->qz;
  return gemm(h, g, s);
}

int vasr_split_tf32(const float* w_dev, float* split_dev, int64_t numel, void* stream) {
  if (!w_dev || !split_dev || numel < 0) return fail(VASR_ERR_INVALID, "null argument");
  KL(launch_split_tf32(w_dev, split_dev, numel, static_cast<cudaStream_t>(stream)));
  return VASR_OK;
}

int vasr_linear_tc(const float* x_dev, int64_t ldx, const float* w_dev, const float* w_split_dev,
                   const float* bias_dev, const float* resid_dev, int64_t ldr, float* out_dev, int64_t ldo, int64_t M,
                   int64_t K, int64_t N, int act, void* stream) {
  if (!x_dev || (!w_dev && !w_split_dev) || !out_dev) return fail(VASR_ERR_INVALID, "null argument");
  if (act < 0 || act > 3) return fail(VASR_ERR_INVALID, "unknown activation");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int dev = 0, sms = 148;
  CK(cudaGetDevice(&dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  GemmArgs g;
  g.A = x_dev; g.lda = ldx; g.W = w_dev; g.bias = bias_dev; g.C = out_dev; g.ldc = ldo;
  g.M = M; g.N = N; g.K = K; g.act = act; g.act_from = 0;
  g.resid = resid_dev; g.ldr = ldr;
  float* hl = nullptr;
  if (!w_split_dev) {       // split on the fly (one extra pass over the weights)
    CK(cudaMallocAsync(reinterpret_cast<void**>(&hl), (size_t)2 * N * K * sizeof(float), s));
    KL(launch_split_tf32(w_dev, hl, N * K, s));
    w_split_dev = hl;
  }
  g.W_split = w_split_dev;
  cudaError_t e = launch_gemm_tc(g, sms, s, nullptr);
  if (hl) CK(cudaFreeAsync(hl, s));
  if (e == cudaErrorNotSupported) return fail(VASR_ERR_UNSUPPORTED, "tensor map could not be encoded for this view");
  if (e != cudaSuccess) return fail(VASR_ERR_CUDA, std::string("launch_gemm_tc: ") + cudaGetErrorString(e));
  return VASR_OK;
}

/* debug hook (not in vasr.h): device buffer of 5 x 128 int64 that CTA 0 of the next tensor-core
 * projection launches fills with clock64 at its pipeline events; NULL switches it off. */
int vasr_debug_gemm_trace(long long* dev_buf) {
  g_trace = dev_buf;
  return VASR_OK;
}

/* debug hook (not in vasr.h): one launch_gemm_tc call with every GemmArgs field exposed, for testing the
 * tensor-core projection kernel one instantiation at a time (tests/test_projection_variants.py).  Device arrays are
 * used as given; the module's own parameters (W as nn.Linear stores it, bias, and for the folded LayerNorm its gamma
 * and beta) are host arrays, prepared the way the engine packs them: fold_ln when ln_gamma is set, gate_perm_row on
 * the rows of the unpermuted [gate | local | global] weight when gate is set, then the TF32 split.  num_sms = 0 takes
 * the device's count; 1 selects the single-CTA kernel.  On return `variant` holds the launched instantiation
 * (TcVariant field order; family 0 = nothing launched), and the call has synchronised the stream. */
struct vasr_debug_gemm_args {
  const float* A; int64_t lda, rows_per_batch, batch_stride;
  int64_t M, N, K;
  float* C; int64_t ldc;
  const float* resid; int64_t ldr;
  const float* q_scale; const float* q_zp;
  const float* pe_time; const float* pe_freq; int64_t pe_half, pe_rows;
  float* amax_val; int32_t* amax_idx;
  const float* W; const float* bias; const float* ln_gamma; const float* ln_beta;  // host
  float ln_eps; int32_t act, act_from, gate, num_sms;
  void* stream;
  int32_t variant[8];
};

int vasr_debug_gemm(vasr_debug_gemm_args* a) {
  if (!a || !a->A || !a->W || (!a->C && !a->amax_val) || (a->ln_gamma && !a->ln_beta))
    return fail(VASR_ERR_INVALID, "null argument");
  const int64_t M = a->M, N = a->N, K = a->K;
  if (M < 0 || N <= 0 || K <= 0) return fail(VASR_ERR_INVALID, "bad shape");
  if (a->act < 0 || a->act > 3) return fail(VASR_ERR_INVALID, "unknown activation");
  memset(a->variant, 0, sizeof(a->variant));
  cudaStream_t s = static_cast<cudaStream_t>(a->stream);
  std::vector<float> W(a->W, a->W + N * K), b, cs;
  if (a->bias) b.assign(a->bias, a->bias + N);
  const bool lna = a->ln_gamma != nullptr;
  if (lna) {
    std::vector<float> Wf, bf;
    fold_ln(W, N, K, a->bias, a->ln_gamma, a->ln_beta, &Wf, &bf, &cs);
    W.swap(Wf);
    b.swap(bf);
  }
  if (a->gate && N % 192 == 0) {    // other widths: launch_gemm_tc declines the gate epilogue
    std::vector<float> Wp(W.size()), bp(b.size());
    for (int64_t rp = 0; rp < N; ++rp) {
      const int r = gate_perm_row((int)rp, (int)(N / 3));
      memcpy(&Wp[(size_t)rp * K], &W[(size_t)r * K], (size_t)K * sizeof(float));
      if (!b.empty()) bp[(size_t)rp] = b[(size_t)r];
    }
    W.swap(Wp);
    b.swap(bp);
  }
  // one scratch allocation: W | W_split | bias | ln_s | ln_stats, each 16-byte aligned
  auto al4 = [](int64_t n) { return (n + 3) & ~(int64_t)3; };
  const int64_t o_ws = al4(N * K), o_b = o_ws + al4(2 * N * K), o_s = o_b + al4(N), o_st = o_s + al4(N);
  const int64_t total = o_st + al4(2 * (M > 0 ? M : 1));
  float* buf = nullptr;
  CK(cudaMallocAsync(reinterpret_cast<void**>(&buf), (size_t)total * sizeof(float), s));
  auto put = [&](const std::vector<float>& v, int64_t off) {
    return v.empty() ? cudaSuccess : cudaMemcpyAsync(buf + off, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice, s);
  };
  cudaError_t e = put(W, 0);
  if (e == cudaSuccess) e = put(b, o_b);
  if (e == cudaSuccess) e = put(cs, o_s);
  if (e == cudaSuccess) e = launch_split_tf32(buf, buf + o_ws, N * K, s);
  if (e != cudaSuccess) {
    cudaFreeAsync(buf, s);
    return fail(VASR_ERR_CUDA, std::string("vasr_debug_gemm staging: ") + cudaGetErrorString(e));
  }
  GemmArgs g;
  g.A = a->A; g.lda = a->lda; g.rows_per_batch = a->rows_per_batch; g.batch_stride = a->batch_stride;
  g.W = buf; g.W_split = buf + o_ws; g.bias = b.empty() ? nullptr : buf + o_b;
  g.q_scale = a->q_scale; g.q_zp = a->q_zp;
  g.C = a->C; g.ldc = a->ldc;
  g.M = M; g.N = N; g.K = K;
  g.act = a->act; g.act_from = a->act_from;
  g.resid = a->resid; g.ldr = a->ldr;
  if (lna) { g.ln_s = buf + o_s; g.ln_stats = buf + o_st; g.ln_eps = a->ln_eps; }
  g.amax_val = a->amax_val; g.amax_idx = a->amax_idx;
  g.gate = a->gate;
  g.pe_time = a->pe_time; g.pe_freq = a->pe_freq; g.pe_half = (int)a->pe_half; g.pe_rows = a->pe_rows;
  int sms = a->num_sms;
  if (sms <= 0) {
    int dev = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  tc_last_variant = nullptr;
  e = launch_gemm_tc(g, sms, s, nullptr);
  const TcVariant* v = tc_last_variant;
  if (e == cudaErrorNotSupported) (void)cudaGetLastError();
  cudaFreeAsync(buf, s);
  const cudaError_t se = cudaStreamSynchronize(s);     // a fault of the kernel surfaces here
  if (e == cudaErrorNotSupported) return fail(VASR_ERR_UNSUPPORTED, "launch_gemm_tc declines this projection");
  if (e != cudaSuccess) return fail(VASR_ERR_CUDA, std::string("launch_gemm_tc: ") + cudaGetErrorString(e));
  if (se != cudaSuccess) return fail(VASR_ERR_CUDA, std::string("vasr_debug_gemm: ") + cudaGetErrorString(se));
  if (v) {
    const int f[8] = {v->family, v->tn, v->act, v->pe, v->resid, v->quant, v->wres, v->epi};
    memcpy(a->variant, f, sizeof(f));
  }
  return VASR_OK;
}

/* debug hook (not in vasr.h): one call of a streaming kernel's launcher from kernels.cuh, for testing it on its own
 * (tests/test_stream_kernels.py).  `kernel` names the launcher; each takes the fields its comment lists, as device
 * pointers, and ignores the others:
 *   layer_norm     x, ldx, y, ldy, gamma, beta, M, C
 *   ln_dwconv      x, y (= u), gamma, beta, w, bias, B, L, C, k, run_len (0: the launcher's rule; the run length
 *                  used comes back in run_len_used)
 *   adaptive_pool  x, ldx, y, B, L, K, C, rag, f_in, f_out
 *   attention      x (= q), ldx, kv, y (= o), ldy, B, L, K (= keys), heads, hd, rag
 *   gate_mix       x (= f3), y, M, C
 *   argmax         x (= logits), pred, M, V
 *   ctc_collapse   pred, tokens, lens, B, L, blank, collapse, rag, and with amax_val: amax_idx, slots
 *   ctc_runs       pred, tokens, starts, ends, lens, B, L, blank
 *   minmax         x, ldx, M, c0, nc, mm, then set_qparams into q_scale / q_zp
 * The call synchronises the stream; a launcher that declines its arguments gives VASR_ERR_UNSUPPORTED. */
struct vasr_debug_kernel_args {
  const char* kernel;
  const float* x; int64_t ldx;
  const float* kv;
  float* y; int64_t ldy;
  const float* gamma; const float* beta; const float* w; const float* bias;
  int32_t* pred; int32_t* tokens; int32_t* lens; int32_t* starts; int32_t* ends;
  const float* amax_val; const int32_t* amax_idx; int32_t slots;
  float* mm; float* q_scale; float* q_zp; int32_t c0, nc;
  const int32_t* rag; int32_t f_in, f_out;
  int64_t B, L, M, K;
  int32_t C, k, heads, hd, V, blank, collapse, run_len;
  void* stream;
  int32_t run_len_used;
};

int vasr_debug_kernel(vasr_debug_kernel_args* a) {
  if (!a || !a->kernel) return fail(VASR_ERR_INVALID, "null argument");
  const std::string n(a->kernel);
  cudaStream_t s = static_cast<cudaStream_t>(a->stream);
  cudaError_t e;
  if (n == "layer_norm") {
    e = launch_layer_norm(a->x, a->ldx, a->y, a->ldy, a->gamma, a->beta, a->M, a->C, s, nullptr);
  } else if (n == "ln_dwconv") {
    int used = 0;
    e = launch_ln_dwconv(a->x, a->y, a->gamma, a->beta, a->w, a->bias, a->B, a->L, a->C, a->k, s, nullptr, a->run_len,
                         &used);
    a->run_len_used = used;
  } else if (n == "adaptive_pool") {
    e = launch_adaptive_pool(a->x, a->ldx, a->y, a->B, a->L, a->K, a->C, s, nullptr, a->rag, a->f_in, a->f_out);
  } else if (n == "attention") {
    e = launch_attention(a->x, a->ldx, a->kv, a->y, a->ldy, a->B, a->L, a->K, a->heads, a->hd, s, nullptr, a->rag);
  } else if (n == "gate_mix") {
    e = launch_gate_mix(a->x, a->y, a->M, a->C, s, nullptr);
  } else if (n == "argmax") {
    e = launch_argmax(a->x, a->pred, a->M, a->V, s, nullptr);
  } else if (n == "ctc_collapse") {
    e = launch_ctc_collapse(a->pred, a->tokens, a->lens, a->B, a->L, a->blank, a->collapse, s, nullptr, a->rag,
                            a->amax_val, a->amax_idx, a->slots);
  } else if (n == "ctc_runs") {
    e = launch_ctc_runs(a->pred, a->tokens, a->starts, a->ends, a->lens, a->B, a->L, a->blank, s, nullptr);
  } else if (n == "minmax") {
    e = launch_minmax(a->x, a->ldx, a->M, a->c0, a->nc, a->mm, s, nullptr);
    if (e == cudaSuccess) e = launch_set_qparams(a->mm, a->q_scale, a->q_zp, a->c0, a->nc, s, nullptr);
  } else {
    return fail(VASR_ERR_INVALID, "unknown kernel: " + n);
  }
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    return fail(e == cudaErrorInvalidValue ? VASR_ERR_UNSUPPORTED : VASR_ERR_CUDA,
                "launch_" + n + ": " + cudaGetErrorString(e));
  }
  const cudaError_t se = cudaStreamSynchronize(s);     // a fault of the kernel surfaces here
  if (se != cudaSuccess) return fail(VASR_ERR_CUDA, "vasr_debug_kernel " + n + ": " + cudaGetErrorString(se));
  return VASR_OK;
}

/* debug hook (not in vasr.h): prints and clears the per-shape projection timings gathered under VASR_PROF=1 */
int vasr_debug_dump_profile(vasr_handle* h) {
  if (!h) return fail(VASR_ERR_INVALID, "null handle");
  CK(cudaDeviceSynchronize());
  std::unordered_map<std::string, std::pair<int, float>> agg;
  float total = 0.f;
  for (auto& pe : h->prof_ev) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, pe.e0, pe.e1);
    auto& a = agg[pe.tag];
    a.first += 1;
    a.second += ms;
    total += ms;
    cudaEventDestroy(pe.e0);
    cudaEventDestroy(pe.e1);
  }
  h->prof_ev.clear();
  for (auto& kv : agg)
    printf("%-44s x%3d  total %8.3f ms  avg %7.1f us\n", kv.first.c_str(), kv.second.first, kv.second.second,
           1e3f * kv.second.second / kv.second.first);
  printf("projections total %.3f ms\n", total);
  fflush(stdout);
  return VASR_OK;
}

int64_t vasr_tc_launches(const vasr_handle* h) { return h ? h->tc_launches : 0; }
int64_t vasr_kernel_launches(const vasr_handle* h) { return h ? h->launches : 0; }
int64_t vasr_workspace_bytes(const vasr_handle* h) { return h ? (int64_t)h->ws.bytes : 0; }

int vasr_set_timing(vasr_handle* h, int enabled) {
  if (!h) return fail(VASR_ERR_INVALID, "null handle");
  h->timing = enabled != 0;
  return VASR_OK;
}

int vasr_last_timing(const vasr_handle* h, float* scan_ms, int32_t* scan_launches, float* total_ms) {
  if (!h) return fail(VASR_ERR_INVALID, "null handle");
  if (!h->ev_total) return fail(VASR_ERR_STATE, "timing was not enabled for the last call");
  CK(cudaEventSynchronize(h->ev_t1));
  float tot = 0.f, sc = 0.f;
  CK(cudaEventElapsedTime(&tot, h->ev_t0, h->ev_t1));
  for (int i = 0; i + 1 < h->ev_used; i += 2) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->ev[i], h->ev[i + 1]));
    sc += ms;
  }
  if (scan_ms) *scan_ms = sc;
  if (scan_launches) *scan_launches = h->ev_used / 2;
  if (total_ms) *total_ms = tot;
  return VASR_OK;
}

}  // extern "C"
