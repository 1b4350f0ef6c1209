// scan.cu — selective scan (SelectiveSSM._sequential_scan / _mamba_scan / _parallel_scan,
// velocity_asr/ssm.py:134-337), with the D skip (ssm.py:170,213) and the silu(z) gate
// (ssm.py:129) fused into the same pass.
//
//   h[d,n] <- exp(dt[t,d] A[n]) h[d,n] + x[t,d] dt[t,d] B[t,n];   y[t,d] = sum_n h[d,n] C[t,n] + x[t,d] D[d]
//
// Mapping.  A (b, d) row is sequential in t and is owned by LPR = N/8 lanes of one warp; each
// lane keeps 8 states in registers as four packed fp32x2 values, so the whole update runs on
// FFMA2/FMUL2 (two state updates per issue slot).  The partial dot products <h, C> of eight
// consecutive timesteps are reduced across the LPR lanes with one transpose-reduce (7 shuffles
// per 8 steps for N = 64 instead of 24), which leaves each lane holding the finished y of one
// (or two) timesteps: that lane applies the D skip and the gate.  All rows of a CTA belong to
// one utterance, so the B/C rows of a 32-step chunk are staged once in shared memory and read
// by every row as broadcast 16-byte loads; x/dt/z/y tiles go through shared memory too so
// global accesses are contiguous runs per timestep.
//
// Structured A.  The reference never re-initialises A_log (model.py:305-318), so A[n] = -(n+1)
// in every random-init model (ssm.py:83-84).  Then exp(dt A[n]) = r^(n+1) with r = exp(-dt):
// two MUFU ops per lane-step plus a packed multiply chain instead of one MUFU per state.
// The generic path (one ex2 per state) is kept for trained checkpoints.
//
// 'parallel' quirk.  The reference's default scan (ssm.py:228-295) is an exclusive scan with a
// mis-ordered down-sweep combine.  It equals (SURVEY.md section 5.7, oracle/velocity_oracle.py
// scan_parallel_streaming), with H[e] the true state after e steps, S[e] = sum_{s<e} dt_s and
// parent(t) = t & (t-1):
//     hP[0] = 0;  hP[t] = hP[parent] + exp(A S[t]) * (H[t] - exp(A (S[t]-S[parent])) H[parent])
// which is evaluated left to right with O(log L) saved ancestors per state.
#include <cstdlib>
#include <map>
#include <mutex>
#include <utility>

#include "common.cuh"
#include "kernels.cuh"

namespace vasr {

namespace {

constexpr int SPL = 8;             // states per lane
constexpr int SCAN_THREADS = 128;
constexpr int NLEV = 26;           // ancestor levels of the quirk mode (L < 2^24)
constexpr float LOG2E = 1.4426950408889634f;

struct State8 {
  u64 v[4];
};

// p[k] = r^(n0 + k + 1), r = 2^s  (s = -dt * log2 e)
__device__ __forceinline__ void powers_structured(float s, float n0p1, State8& p) {
  const float r1 = ex2_approx(s);
  const float e1 = ex2_approx(s * n0p1);
  const float r2 = r1 * r1;
  const u64 rr = pack2(r2, r2);
  p.v[0] = pack2(e1, e1 * r1);
  p.v[1] = mul2(p.v[0], rr);
  p.v[2] = mul2(p.v[1], rr);
  p.v[3] = mul2(p.v[2], rr);
}
// p[k] = 2^(s * al2[k]),  al2[k] = A[n0+k] * log2 e  (negative), s = dt >= 0
__device__ __forceinline__ void powers_generic(float s, const float (&al2)[SPL], State8& p) {
#pragma unroll
  for (int k = 0; k < 4; ++k) p.v[k] = pack2(ex2_approx(s * al2[2 * k]), ex2_approx(s * al2[2 * k + 1]));
}

// ------------------------------------------------------------------------------------------
// The reference's 'parallel' scan (quirk).  One row per lane group (8 states per lane).  Steps are
// taken eight at a time, aligned to multiples of 8, so the ancestor an index needs is known at
// compile time for seven of the eight steps:  parent(8q+i) = 8q + (i & (i-1)).  Ancestor levels
// 1..3 ("most recent index with at least l trailing zeros") therefore live in registers; only the
// step at 8q touches the higher levels, which sit in local memory (one read, ~one write per 8 steps).
//
// Where the quirk stops costing anything.  Every term that enters hP[t] carries the factor exp(A S[t]), the decay
// from time 0, and S only grows (dt is a softplus output, ssm.py:118).  Once min_n |A[n]| S[t] log2(e) >= 127 that
// factor is exactly 0 for every state in this kernel's arithmetic (ex2.approx.ftz flushes results below 2^-126;
// the reference's fp32 product of dA is below 1e-38 there, i.e. invisible), so hP[t] = hP[parent(t)] bit for bit
// from then on, and the true state H is never needed again:
//   phase 1  (until every row of the CTA has passed that point, checked once per 16-step chunk): the full rule;
//   phase 2  (from there to the next power of two P2): hP[t] = hP[parent(t)], y = <hP[t], C[t]> + x D — one FMA
//            per state, no B, no dt;
//   phase 3  (t >= P2): every ancestor of t is >= P2 or 0, so hP[t] = hP[0] = 0 and y = x D (gated): a plain
//            streaming pass over x and z.
// Phases 2 and 3 are shortcuts of phase 1, not approximations: the full rule computes the same bits (it multiplies
// by an exact zero), so a row's result does not depend on its CTA mates or on where the switch falls.  With the
// reference's random-init weights dt ~ 0.7 and the switch comes after ~150 of config 2's 751 tokens; a model whose
// dt stays small (sum of dt below ~110 over the utterance) runs phase 1 throughout.
// ------------------------------------------------------------------------------------------
constexpr int TCQ = 16;
constexpr float QUIRK_DEAD_LOG2 = 127.0f;     // 2^-127: below the smallest normal fp32, ex2.approx.ftz returns exactly 0

struct Anc {
  State8 hp, H;
  double S;
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N_) : "memory"); }

// State of the narrow mode: two states per lane (one packed pair), see scan_quirk_kernel.
struct Anc1 {
  u64 hp, H;
  double S;
};

template <int LPR, bool STRUCT>
__global__ void __launch_bounds__(SCAN_THREADS) scan_quirk_kernel(ScanArgs a) {
  pdl_wait();
  constexpr int N = LPR * SPL;
  constexpr int ROWS = SCAN_THREADS / LPR;
  constexpr int NR = (LPR == 8) ? 3 : (LPR == 4 ? 2 : (LPR == 2 ? 1 : 0));
  constexpr int TPL = 8 >> NR;
  constexpr int HL = NLEV - 4;   // levels >= 4
  constexpr int NN = 2 * LPR;    // states that stay in the narrow mode: 0 .. NN-1, two per lane

  // two stages: the tiles of chunk c + 1 travel (cp.async) while chunk c is computed.  B / C rows are stored in
  // 16-byte pieces at permuted slots (piece f of a row at slot (f & 1) LPR + (f >> 1)) so that the 16-byte reads
  // of the wide mode hit distinct banks; the narrow mode reads its two states out of the same layout.
  __shared__ __align__(16) float sBs[2][TCQ][N];
  __shared__ __align__(16) float sCs[2][TCQ][N];
  __shared__ __align__(16) float sxs[2][TCQ][ROWS];
  __shared__ __align__(16) float sdts[2][TCQ][ROWS];
  __shared__ __align__(16) float szs[2][TCQ][ROWS];
  __shared__ float sy[TCQ][ROWS];

  const int tid = threadIdx.x;
  const int rl = tid / LPR, j = tid % LPR;
  const int n0 = j * SPL;
  const int d0 = blockIdx.x * ROWS;
  const int64_t b = blockIdx.y;
  const int64_t L = a.L;
  const bool gate = a.z != nullptr;

  float al2[SPL];
#pragma unroll
  for (int k = 0; k < SPL; ++k) al2[k] = a.A[n0 + k] * LOG2E;
  const float n0p1 = (float)(n0 + 1);
  const float Dd = a.D ? a.D[d0 + rl] : 0.f;
  float amin_l2 = 3.0e38f;                    // min_n |A[n]| log2 e: the slowest-decaying state
#pragma unroll
  for (int k = 0; k < SPL; ++k) amin_l2 = fminf(amin_l2, fabsf(al2[k]));
#pragma unroll
  for (int o = 1; o < LPR; o <<= 1) amin_l2 = fminf(amin_l2, __shfl_xor_sync(0xffffffffu, amin_l2, o));
  bool frozen = false;                        // phase 2: hP[t] = hP[parent(t)]
  int64_t t_zero = L;                         // phase 3 starts here (a power of two >= the start of phase 2)
  // Narrow mode (structured A): the states decay in order, state n at the rate (n + 1).  Once exp(A[n] S) is an
  // exact zero for every n >= NN in every row of the CTA, and the next power of two has passed (so that their
  // hP is zero, not just frozen), only the NN slowest states are left: the CTA continues with two states per lane
  // instead of eight.  With dt ~ 0.7 that is after the first 16 tokens.  What it drops is exact zeros, but its powers
  // (r^(2j+1) directly) and the order of its state sum differ from the wide mode's: unlike phases 2 and 3, the switch
  // can move the last bit of a row's state sum (DESIGN.md).
  int64_t t_narrow = L;
  bool narrow_known = !STRUCT || N <= NN;

  Anc cur, a1, a2, a3;
#pragma unroll
  for (int k = 0; k < 4; ++k) cur.hp.v[k] = cur.H.v[k] = 0ull;
  cur.S = 0.0;
  a1 = a2 = a3 = cur;
  float hi_hp[HL][SPL], hi_H[HL][SPL];
  double hi_S[HL];
  // only the levels an index below L can reach are ever read (index 8q with z trailing zeros reads level
  // z + 1 = entry z - 3, and 2^z < L).  These arrays are indexed dynamically, i.e. they live in local memory;
  // clearing all 22 of them cost a short sequence — the global branch runs L = 93 — more than its 93 steps.
  int hl_used = 0;
  while (hl_used < HL && (1LL << (hl_used + 3)) < a.L) ++hl_used;
  for (int l = 0; l < hl_used; ++l) {
    hi_S[l] = 0.0;
#pragma unroll
    for (int k = 0; k < SPL; ++k) hi_hp[l][k] = hi_H[l][k] = 0.f;
  }

  // ---- pieces shared by the wide and the narrow chunk loop
  // 16-byte cp.async needs 16-byte aligned rows everywhere; anything else is staged through registers, chunk by chunk
  const bool async_ok = !((a.ldx | a.lddt | a.ldb | a.ldc | (gate ? a.ldz : 0)) & 3) &&
                        !((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.dt) |
                           reinterpret_cast<uintptr_t>(a.Bm) | reinterpret_cast<uintptr_t>(a.Cm) |
                           (gate ? reinterpret_cast<uintptr_t>(a.z) : 0)) & 15);
  // tiles of the chunk starting at t0 -> stage st.  nstates: how many leading states of B / C are wanted.
  // Asynchronous form: always ends with a commit (an empty group past the end of the sequence).
  auto load_chunk = [&](int64_t t0, int st, int nstates, bool async) {
    const int tcn = t0 >= L ? 0 : (int)((L - t0) < TCQ ? (L - t0) : TCQ);
    const int nf = nstates / 4;
    for (int idx = tid; idx < TCQ * nf; idx += SCAN_THREADS) {
      const int t = idx / nf, f = idx % nf;
      if (t >= tcn) continue;
      const int64_t row = b * L + t0 + t;
      const int slot = (f & 1) * LPR + (f >> 1);
      if (async) {
        if (!frozen) cp_async16(&sBs[st][t][4 * slot], a.Bm + row * a.ldb + 4 * f);
        cp_async16(&sCs[st][t][4 * slot], a.Cm + row * a.ldc + 4 * f);
      } else {
        float vb[4] = {0.f, 0.f, 0.f, 0.f}, vc[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (!frozen) vb[i] = __ldg(a.Bm + row * a.ldb + 4 * f + i);
          vc[i] = __ldg(a.Cm + row * a.ldc + 4 * f + i);
        }
        *reinterpret_cast<float4*>(&sBs[st][t][4 * slot]) = make_float4(vb[0], vb[1], vb[2], vb[3]);
        *reinterpret_cast<float4*>(&sCs[st][t][4 * slot]) = make_float4(vc[0], vc[1], vc[2], vc[3]);
      }
    }
    if (async) {
      for (int idx = tid; idx < TCQ * (ROWS / 4); idx += SCAN_THREADS) {
        const int t = idx / (ROWS / 4), r = 4 * (idx % (ROWS / 4));
        if (t >= tcn) continue;
        const int64_t row = b * L + t0 + t;
        cp_async16(&sxs[st][t][r], a.x + row * a.ldx + d0 + r);
        if (!frozen) cp_async16(&sdts[st][t][r], a.dt + row * a.lddt + d0 + r);
        if (gate) cp_async16(&szs[st][t][r], a.z + row * a.ldz + d0 + r);
      }
      cp_async_commit();
    } else {
      for (int idx = tid; idx < TCQ * ROWS; idx += SCAN_THREADS) {
        const int t = idx / ROWS, r = idx % ROWS;
        if (t >= tcn) continue;
        const int64_t row = b * L + t0 + t;
        sxs[st][t][r] = __ldg(a.x + row * a.ldx + d0 + r);
        if (!frozen) sdts[st][t][r] = __ldg(a.dt + row * a.lddt + d0 + r);
        if (gate) szs[st][t][r] = __ldg(a.z + row * a.ldz + d0 + r);
      }
    }
  };
  // top of a chunk: request the next chunk's tiles, make this chunk's visible; returns this chunk's stage
  auto begin_chunk = [&](int64_t tc0, int nstates) {
    const int st = (int)((tc0 / TCQ) & 1);
    if (async_ok) {
      load_chunk(tc0 + TCQ, st ^ 1, nstates, true);   // everyone left that stage at the previous end_chunk barrier
      cp_async_wait<1>();
    } else {
      load_chunk(tc0, st, nstates, false);
    }
    __syncthreads();
    return st;
  };
  if (async_ok) load_chunk(0, 0, N, true);
  auto reduce_gate = [&](float (&yp)[8], int g8, const float (*sx)[ROWS], const float (*sz)[ROWS]) {   // 8 steps' partial <hP, C> -> sy
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      const int lane_bit = LPR >> (r + 1);
      const int cnt = 4 >> r;
      const bool hi = (j & lane_bit) != 0;
#pragma unroll
      for (int i = 0; i < cnt; ++i) {
        const float mine = hi ? yp[i + cnt] : yp[i];
        const float other = hi ? yp[i] : yp[i + cnt];
        yp[i] = mine + __shfl_xor_sync(0xffffffffu, other, lane_bit);
      }
    }
#pragma unroll
    for (int i = 0; i < TPL; ++i) {
      const int t = g8 + j * TPL + i;
      float yv = yp[i] + sx[t][rl] * Dd;
      if (gate) {
        const float zv = sz[t][rl];
        yv *= zv / (1.0f + __expf(-zv));
      }
      sy[t][rl] = yv;
    }
  };
  // end of a chunk: phase switch (has every row of the CTA decayed to an exact zero?) and the stores
  auto end_chunk = [&](int64_t tc0, int tcn, double S_row) {
    const bool dead = frozen || (float)S_row * amin_l2 >= QUIRK_DEAD_LOG2;
    const bool all_dead = __syncthreads_and(dead) != 0;       // also orders sy before the stores below
    if (all_dead && !frozen) {
      frozen = true;
      int64_t p2 = TCQ;
      while (p2 < tc0 + TCQ) p2 <<= 1;
      t_zero = p2;
    }
    for (int idx = tid; idx < tcn * ROWS; idx += SCAN_THREADS) {
      const int t = idx / ROWS, r = idx % ROWS;
      a.y[(b * L + tc0 + t) * a.ldy + d0 + r] = sy[t][r];
    }
  };

  // =========================================================================== wide mode: 8 states per lane
  int64_t tc0 = 0;
  for (; tc0 < L && tc0 < t_zero && tc0 < t_narrow; tc0 += TCQ) {
    if (tc0 + TCQ >= L) pdl_trigger();     // last chunk: see scan_seq_kernel
    const int tcn = (int)((L - tc0) < TCQ ? (L - tc0) : TCQ);
    const int st = begin_chunk(tc0, N);
    float (*sB)[N] = sBs[st];
    float (*sC)[N] = sCs[st];
    float (*sx)[ROWS] = sxs[st];
    float (*sdt)[ROWS] = sdts[st];
    float (*sz)[ROWS] = szs[st];

#pragma unroll 1
    for (int g8 = 0; g8 < TCQ; g8 += 8) {
      if (g8 >= tcn) break;
      float yp[8];
      // one step: hP from `par`, output partial, then the true-recurrence update of cur.H / cur.S
      auto step = [&](int i, const Anc& par, bool has_parent) {
        const int t = g8 + i;
        const ulonglong2 c01 = *reinterpret_cast<const ulonglong2*>(&sC[t][4 * j]);
        const ulonglong2 c23 = *reinterpret_cast<const ulonglong2*>(&sC[t][4 * (LPR + j)]);
        if (has_parent && frozen) {
#pragma unroll
          for (int k = 0; k < 4; ++k) cur.hp.v[k] = par.hp.v[k];
        } else if (has_parent) {
          const float Sf = (float)cur.S;
          const float dS = (float)(cur.S - par.S);
          State8 q, pd;
          if (STRUCT) {
            powers_structured(-Sf * LOG2E, n0p1, q);
            powers_structured(-dS * LOG2E, n0p1, pd);
          } else {
            powers_generic(Sf, al2, q);
            powers_generic(dS, al2, pd);
          }
          const u64 neg1 = pack2(-1.f, -1.f);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const u64 inner = fma2(mul2(pd.v[k], neg1), par.H.v[k], cur.H.v[k]);   // H - pd * H[parent]
            cur.hp.v[k] = fma2(q.v[k], inner, par.hp.v[k]);
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) cur.hp.v[k] = 0ull;
        }
        u64 acc = fma2(cur.hp.v[1], c01.y, mul2(cur.hp.v[0], c01.x));
        u64 acc2 = fma2(cur.hp.v[3], c23.y, mul2(cur.hp.v[2], c23.x));
        yp[i] = hsum2(add2(acc, acc2));
      };
      auto advance = [&](int i) {
        if (frozen) return;                   // H and S feed nothing any more
        const int t = g8 + i;
        const float dtv = sdt[t][rl];
        State8 p;
        if (STRUCT) powers_structured(-dtv * LOG2E, n0p1, p);
        else powers_generic(dtv, al2, p);
        const float u = sx[t][rl] * dtv;
        const u64 uu = pack2(u, u);
        const ulonglong2 b01 = *reinterpret_cast<const ulonglong2*>(&sB[t][4 * j]);
        const ulonglong2 b23 = *reinterpret_cast<const ulonglong2*>(&sB[t][4 * (LPR + j)]);
        cur.H.v[0] = fma2(p.v[0], cur.H.v[0], mul2(uu, b01.x));
        cur.H.v[1] = fma2(p.v[1], cur.H.v[1], mul2(uu, b01.y));
        cur.H.v[2] = fma2(p.v[2], cur.H.v[2], mul2(uu, b23.x));
        cur.H.v[3] = fma2(p.v[3], cur.H.v[3], mul2(uu, b23.y));
        cur.S += (double)dtv;
      };

      // ---- i = 0 : index 8q, ancestor level >= 4 (dynamic)
      {
        const int64_t tg = tc0 + g8;
        if (tg == 0) {
          step(0, cur, false);
        } else {
          const int z = 3 + (__ffsll((long long)(tg >> 3)) - 1);
          const int pl = z + 1 - 4;
          Anc par;
          par.S = hi_S[pl];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            par.hp.v[k] = pack2(hi_hp[pl][2 * k], hi_hp[pl][2 * k + 1]);
            par.H.v[k] = pack2(hi_H[pl][2 * k], hi_H[pl][2 * k + 1]);
          }
          step(0, par, true);
          for (int l = 4; l <= z; ++l) {
            hi_S[l - 4] = cur.S;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              unpack2(cur.hp.v[k], hi_hp[l - 4][2 * k], hi_hp[l - 4][2 * k + 1]);
              unpack2(cur.H.v[k], hi_H[l - 4][2 * k], hi_H[l - 4][2 * k + 1]);
            }
          }
          a1 = a2 = a3 = cur;
        }
        advance(0);
      }
      step(1, a1, true); advance(1);
      step(2, a2, true); a1 = cur; advance(2);
      step(3, a1, true); advance(3);
      step(4, a3, true); a1 = a2 = cur; advance(4);
      step(5, a1, true); advance(5);
      step(6, a2, true); a1 = cur; advance(6);
      step(7, a1, true); advance(7);
      reduce_gate(yp, g8, sx, sz);
    }
    if (!narrow_known && !frozen) {          // are the states >= NN exact zeros in every row from here on?
      const bool hi_dead = (float)cur.S * ((float)(NN + 1) * LOG2E) >= QUIRK_DEAD_LOG2;
      if (__syncthreads_and(hi_dead)) {
        narrow_known = true;
        int64_t p2 = TCQ;
        while (p2 < tc0 + TCQ) p2 <<= 1;
        t_narrow = p2;
      }
    }
    end_chunk(tc0, tcn, cur.S);
  }

  // =========================================================================== narrow mode: 2 states per lane
  if (STRUCT && tc0 < L && tc0 < t_zero && !frozen) {
    // states 2 j, 2 j + 1 of the row: pair (j % 4) of the lane that held states 8 (j / 4) ...; S is shared.
    // Ancestors: tc0 is a power of two, so every index from here on has its ancestors at or after tc0, or at 0
    // (state zero): the saved levels start again from zero, only the true state and S carry over.
    Anc1 c1, b1, b2, b3;
    {
      const int src = (tid & 31) - j + (j >> 2);
      u64 mine = 0ull;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const u64 v = __shfl_sync(0xffffffffu, cur.H.v[k], src);
        if (k == (j & 3)) mine = v;
      }
      c1.H = mine;
      c1.hp = 0ull;
      c1.S = cur.S;
      b1 = b2 = b3 = c1;
    }
    for (int l = 0; l < hl_used; ++l) {
      hi_S[l] = 0.0;
      hi_hp[l][0] = hi_hp[l][1] = hi_H[l][0] = hi_H[l][1] = 0.f;
    }
    const float e_mul = (float)(2 * j + 1);
    auto pw = [&](float s) {                 // (r^(2j+1), r^(2j+2)), r = 2^s
      const float r1 = ex2_approx(s);
      const float e1 = ex2_approx(s * e_mul);
      return pack2(e1, e1 * r1);
    };
    for (; tc0 < L && tc0 < t_zero; tc0 += TCQ) {
      if (tc0 + TCQ >= L) pdl_trigger();
      const int tcn = (int)((L - tc0) < TCQ ? (L - tc0) : TCQ);
      const int st = begin_chunk(tc0, NN);             // only the first NN states of B / C travel from here on
      float (*sB)[N] = sBs[st];
      float (*sC)[N] = sCs[st];
      float (*sx)[ROWS] = sxs[st];
      float (*sdt)[ROWS] = sdts[st];
      float (*sz)[ROWS] = szs[st];
      // states 2 j, 2 j + 1 inside the permuted 16-byte pieces: piece j / 2, second half for odd j
      const int nsl = 4 * (((j >> 1) & 1) * LPR + (j >> 2)) + 2 * (j & 1);
#pragma unroll 1
      for (int g8 = 0; g8 < TCQ; g8 += 8) {
        if (g8 >= tcn) break;
        float yp[8];
        auto step = [&](int i, const Anc1& par) {
          const int t = g8 + i;
          if (frozen) {
            c1.hp = par.hp;
          } else {
            const u64 q = pw(-(float)c1.S * LOG2E);
            const u64 pd = pw(-(float)(c1.S - par.S) * LOG2E);
            const u64 inner = fma2(mul2(pd, pack2(-1.f, -1.f)), par.H, c1.H);
            c1.hp = fma2(q, inner, par.hp);
          }
          yp[i] = hsum2(mul2(c1.hp, *reinterpret_cast<const u64*>(&sC[t][nsl])));
        };
        auto advance = [&](int i) {
          if (frozen) return;
          const int t = g8 + i;
          const float dtv = sdt[t][rl];
          const float u = sx[t][rl] * dtv;
          c1.H = fma2(pw(-dtv * LOG2E), c1.H, mul2(pack2(u, u), *reinterpret_cast<const u64*>(&sB[t][nsl])));
          c1.S += (double)dtv;
        };
        {
          const int64_t tg = tc0 + g8;                 // > 0 here
          const int z = 3 + (__ffsll((long long)(tg >> 3)) - 1);
          const int pl = z + 1 - 4;
          Anc1 par;
          par.S = hi_S[pl];
          par.hp = pack2(hi_hp[pl][0], hi_hp[pl][1]);
          par.H = pack2(hi_H[pl][0], hi_H[pl][1]);
          step(0, par);
          for (int l = 4; l <= z; ++l) {
            hi_S[l - 4] = c1.S;
            unpack2(c1.hp, hi_hp[l - 4][0], hi_hp[l - 4][1]);
            unpack2(c1.H, hi_H[l - 4][0], hi_H[l - 4][1]);
          }
          b1 = b2 = b3 = c1;
          advance(0);
        }
        step(1, b1); advance(1);
        step(2, b2); b1 = c1; advance(2);
        step(3, b1); advance(3);
        step(4, b3); b1 = b2 = c1; advance(4);
        step(5, b1); advance(5);
        step(6, b2); b1 = c1; advance(6);
        step(7, b1); advance(7);
        reduce_gate(yp, g8, sx, sz);
      }
      end_chunk(tc0, tcn, c1.S);
    }
  }
  cp_async_wait<0>();                       // a tile requested ahead may still be in flight
  // phase 3: hP = 0 for every remaining t, y = x D (gated)
  if (tc0 < L) {
    pdl_trigger();
    auto one = [&](float xv, float dv, float zv) {            // the same operations as the chunk loop with yp = 0
      float yv = 0.f + xv * dv;
      if (gate) yv *= zv / (1.0f + __expf(-zv));
      return yv;
    };
    const bool vec = !((a.ldx | a.ldy | (gate ? a.ldz : 0)) & 3) && !((reinterpret_cast<uintptr_t>(a.x) |
                     reinterpret_cast<uintptr_t>(a.y) | (gate ? reinterpret_cast<uintptr_t>(a.z) : 0)) & 15);
    if (vec) {                   // float4 pieces of a timestep's ROWS values, four independent pieces in flight
      constexpr int RQ = ROWS / 4;
      const int q4 = (tid % RQ) * 4;
      float4 dv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.D) dv = make_float4(a.D[d0 + q4], a.D[d0 + q4 + 1], a.D[d0 + q4 + 2], a.D[d0 + q4 + 3]);
      const int64_t n_t = L - tc0;
      constexpr int TS = SCAN_THREADS / RQ;                    // timesteps covered per pass of the CTA
      for (int64_t t0 = tid / RQ; t0 < n_t; t0 += 4 * TS) {
        float4 xv[4], zv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int64_t t = t0 + u * TS;
          const int64_t row = b * L + tc0 + (t < n_t ? t : t0);
          xv[u] = __ldg(reinterpret_cast<const float4*>(a.x + row * a.ldx + d0 + q4));
          zv[u] = gate ? __ldg(reinterpret_cast<const float4*>(a.z + row * a.ldz + d0 + q4)) : dv;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int64_t t = t0 + u * TS;
          if (t < n_t) {
            const int64_t row = b * L + tc0 + t;
            *reinterpret_cast<float4*>(a.y + row * a.ldy + d0 + q4) =
                make_float4(one(xv[u].x, dv.x, zv[u].x), one(xv[u].y, dv.y, zv[u].y), one(xv[u].z, dv.z, zv[u].z),
                            one(xv[u].w, dv.w, zv[u].w));
          }
        }
      }
    } else {
      for (int64_t idx = tid; idx < (L - tc0) * ROWS; idx += SCAN_THREADS) {
        const int64_t row = b * L + tc0 + idx / ROWS;
        const int r = (int)(idx % ROWS);
        a.y[row * a.ldy + d0 + r] = one(__ldg(a.x + row * a.ldx + d0 + r), a.D ? __ldg(a.D + d0 + r) : 0.f,
                                        gate ? __ldg(a.z + row * a.ldz + d0 + r) : 0.f);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// True recurrence (scan_mode sequential / mamba) for what scan_rp_kernel below does not take: a trained model's
// unstructured A (one ex2 per state), N = 32 / 16, rows that are not 16-byte aligned for its row-pair loads.  It was
// the kernel of every shape until round 2; its structure is the base of scan_rp_kernel.
//
// ncu on the previous version (8 states per lane, register-staged tiles): 115 issued instructions
// per warp-step against 32 packed state operations — index arithmetic of the staging code, the
// 8-lane transpose-reduce and the per-lane power set-up dominated, and the FMA pipe sat at 45 %.
// This version is built to shrink everything that is not a state update:
//   * 16 states per lane, two rows per lane (32 state registers as packed fp32x2): a row is owned by
//     LPR = N/16 lanes, so the set-up cost per row-step (3 MUFU + 6 FMUL), the B/C loads (one
//     16-byte load feeds eight state updates) and the reduction are amortised over twice the work;
//   * B/C/x/dt/z tiles of 16 timesteps arrive by cp.async (LDGSTS) in their NATURAL layout, double
//     buffered: no register staging, no permutation, no per-element address arithmetic.  Lane j
//     reads the float4s j, j+LPR, j+2 LPR, j+3 LPR of a B/C row, i.e. the LPR lanes of a group read
//     consecutive 16-byte pieces (conflict-free) and the lane's states are n = 4 (j + LPR m) + i;
//   * structured A: p[n] = r^(n+1) with r = exp(-dt): the first quad is r^(4j+1) (1, r, r^2, r^3),
//     every further quad is the previous one times r^(4 LPR) — three ex2 per row-step, all other
//     powers are packed multiplies;
//   * the partial dot products of four timesteps x two rows are transpose-reduced over the LPR
//     lanes; the lane that ends up with a finished (t, row pair) applies the D skip and the
//     silu(z) gate and stores the pair straight to global memory (8 bytes per lane, 64 contiguous
//     bytes per timestep per warp).
// ------------------------------------------------------------------------------------------
constexpr int TCH = 16;   // timesteps per staged chunk

template <int LPR, int WARPS, int RPL, bool STRUCT>   // RPL = rows per lane (2 in every instantiation that is built)
__global__ void __launch_bounds__(WARPS * 32, (RPL == 3 ? 256 : RPL == 2 ? 384 : 640) / (WARPS * 32)) scan_seq_kernel(ScanArgs a) {
  pdl_wait();
  constexpr int N = LPR * 16;
  constexpr int GROUPS = 32 / LPR;             // lane groups per warp
  constexpr int ROWS = WARPS * GROUPS * RPL;   // rows per CTA
  constexpr int THREADS = WARPS * 32;
  constexpr int NR = (LPR == 4) ? 2 : (LPR == 2 ? 1 : 0);
  constexpr int NV = 4 * RPL;                  // partials per lane per block of 4 steps
  constexpr int TPL = NV >> NR;                // finished (step, row) values per lane per 4 steps
  constexpr int NF = N / 4, RF = ROWS / 4;     // float4 per B (C) row, per x (dt, z) row
  constexpr int STAGE_FLOATS = TCH * (2 * N + 3 * ROWS);

  extern __shared__ __align__(16) float scan_smem[];
  auto sB = [&](int st) { return scan_smem + st * STAGE_FLOATS; };
  auto sC = [&](int st) { return scan_smem + st * STAGE_FLOATS + TCH * N; };
  auto sX = [&](int st) { return scan_smem + st * STAGE_FLOATS + 2 * TCH * N; };
  auto sDt = [&](int st) { return scan_smem + st * STAGE_FLOATS + 2 * TCH * N + TCH * ROWS; };
  auto sZ = [&](int st) { return scan_smem + st * STAGE_FLOATS + 2 * TCH * N + 2 * TCH * ROWS; };

  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int g = lane / LPR, j = lane % LPR;
  const int rl0 = (warp * GROUPS + g) * RPL;    // first of this lane's rows (within the CTA)
  const int d0 = blockIdx.x * ROWS;
  const int64_t b = blockIdx.y;
  const int64_t L = a.L;
  const bool gate = a.z != nullptr;
  const int nchunks = (int)((L + TCH - 1) / TCH);

  // per-lane exponent constants: exp(dt A[n]) = 2^(dt * A[n] * log2 e)
  float al2[STRUCT ? 1 : 16];
  if (!STRUCT) {
#pragma unroll
    for (int m = 0; m < 4; ++m)
#pragma unroll
      for (int i = 0; i < 4; ++i) al2[4 * m + i] = __ldg(a.A + 4 * (j + LPR * m) + i) * LOG2E;
  }
  const float c_r = -LOG2E;                          // r   = exp(-dt)
  const float c_e = -LOG2E * (float)(4 * j + 1);     // e   = r^(4j+1)
  const float c_q = -LOG2E * (float)(4 * LPR);       // rq  = r^(4 LPR)
  float Dv[RPL];
#pragma unroll
  for (int r = 0; r < RPL; ++r) Dv[r] = a.D ? __ldg(a.D + d0 + rl0 + r) : 0.f;

  u64 H[RPL][8];
#pragma unroll
  for (int r = 0; r < RPL; ++r)
#pragma unroll
    for (int k = 0; k < 8; ++k) H[r][k] = 0ull;

  const float* gB = a.Bm + b * L * a.ldb;
  const float* gC = a.Cm + b * L * a.ldc;
  const float* gX = a.x + b * L * a.ldx + d0;
  const float* gDt = a.dt + b * L * a.lddt + d0;
  const float* gZ = gate ? a.z + b * L * a.ldz + d0 : nullptr;
  float* gY = a.y + b * L * a.ldy + d0 + rl0;

  auto issue = [&](int c) {          // always commits a group (an empty one past the last chunk)
    const int st = c % 3;
    const int64_t tc0 = (int64_t)c * TCH;
    const int tcn = c >= nchunks ? 0 : (int)((L - tc0) < TCH ? (L - tc0) : TCH);
    float* dB = sB(st); float* dC = sC(st); float* dX = sX(st); float* dD = sDt(st); float* dZ = sZ(st);
#pragma unroll
    for (int i = 0; i < (TCH * NF + THREADS - 1) / THREADS; ++i) {
      const int idx = tid + i * THREADS;
      const int t = idx / NF, f = idx % NF;
      if (idx < TCH * NF && t < tcn) {
        cp_async16(dB + t * N + 4 * f, gB + (tc0 + t) * a.ldb + 4 * f);
        cp_async16(dC + t * N + 4 * f, gC + (tc0 + t) * a.ldc + 4 * f);
      }
    }
#pragma unroll
    for (int i = 0; i < (TCH * RF + THREADS - 1) / THREADS; ++i) {
      const int idx = tid + i * THREADS;
      const int t = idx / RF, f = idx % RF;
      if (idx < TCH * RF && t < tcn) {
        cp_async16(dX + t * ROWS + 4 * f, gX + (tc0 + t) * a.ldx + 4 * f);
        cp_async16(dD + t * ROWS + 4 * f, gDt + (tc0 + t) * a.lddt + 4 * f);
        if (gate) cp_async16(dZ + t * ROWS + 4 * f, gZ + (tc0 + t) * a.ldz + 4 * f);
      }
    }
    cp_async_commit();
  };

  // one row, one timestep: advance the 16 states of Hr and return the partial <h, C>
  auto row_step = [&](u64 (&Hr)[8], float dtv, float xv, const ulonglong2 (&bq)[4], const ulonglong2 (&cq)[4]) {
    const float u = xv * dtv;
    const u64 uu = pack2(u, u);
    u64 Pa, Pb, rq2 = 0ull;
    if (STRUCT) {
      const float r = ex2_approx(dtv * c_r);
      const float e = ex2_approx(dtv * c_e);
      const float rq = ex2_approx(dtv * c_q);
      const float r2 = r * r;
      Pa = pack2(e, e * r);
      Pb = mul2(Pa, pack2(r2, r2));
      rq2 = pack2(rq, rq);
    }
    u64 acc0 = 0ull, acc1 = 0ull;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      if (!STRUCT) {
        Pa = pack2(ex2_approx(dtv * al2[4 * m]), ex2_approx(dtv * al2[4 * m + 1]));
        Pb = pack2(ex2_approx(dtv * al2[4 * m + 2]), ex2_approx(dtv * al2[4 * m + 3]));
      }
      Hr[2 * m] = fma2(Pa, Hr[2 * m], mul2(uu, bq[m].x));
      Hr[2 * m + 1] = fma2(Pb, Hr[2 * m + 1], mul2(uu, bq[m].y));
      if (m == 0) {
        acc0 = mul2(Hr[0], cq[0].x);
        acc1 = mul2(Hr[1], cq[0].y);
      } else {
        acc0 = fma2(Hr[2 * m], cq[m].x, acc0);
        acc1 = fma2(Hr[2 * m + 1], cq[m].y, acc1);
      }
      if (STRUCT && m < 3) {
        Pa = mul2(Pa, rq2);
        Pb = mul2(Pb, rq2);
      }
    }
    return hsum2(add2(acc0, acc1));
  };

  // Structured A: the per-row set-up (u, the three ex2 and the first power quad) of step t+1 is computed
  // DURING step t, split in two phases placed between the row updates, so that neither the LDS nor the
  // MUFU latency is ever waited for (warps issue in order: ncu showed the first multiply after the ex2
  // as the top stall of the previous version).
  //
  // One multiply per state is saved by carrying the state SCALED by the input: with h = s_t h' and s_t = u_t,
  //     h'_t = (p_t s_{t-1} / s_t) h'_{t-1} + B_t,     y_t = s_t <h'_t, C_t> + x_t D
  // so the u_t B_t product disappears and the ratio rho = u_{t-1} / u_t is folded into the first power of the
  // chain (two scalar multiplies and one rcp per row-step instead of eight packed multiplies per lane).
  // |u| is kept >= 1e-12 (sign preserved): the perturbation of y is <= 1e-12 |B||C| per step, far below fp32
  // resolution, and it bounds rho so that h' cannot overflow for any |u| < 1e20.
  struct Pre {
    u64 Pa[RPL], Pb[RPL], rq2[RPL];
    float s[RPL];
  };
  auto row_step_pre = [&](u64 (&Hr)[8], u64 Pa, u64 Pb, u64 rq2, float sc, const ulonglong2 (&bq)[4],
                          const ulonglong2 (&cq)[4]) {
    u64 acc0 = 0ull, acc1 = 0ull;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      Hr[2 * m] = fma2(Pa, Hr[2 * m], bq[m].x);
      Hr[2 * m + 1] = fma2(Pb, Hr[2 * m + 1], bq[m].y);
      if (m == 0) {
        acc0 = mul2(Hr[0], cq[0].x);
        acc1 = mul2(Hr[1], cq[0].y);
      } else {
        acc0 = fma2(Hr[2 * m], cq[m].x, acc0);
        acc1 = fma2(Hr[2 * m + 1], cq[m].y, acc1);
      }
      if (m < 3) {
        Pa = mul2(Pa, rq2);
        Pb = mul2(Pb, rq2);
      }
    }
    return sc * hsum2(add2(acc0, acc1));
  };
  float s_carry[RPL];          // scale (= clamped u) of the last step executed
#pragma unroll
  for (int q = 0; q < RPL; ++q) s_carry[q] = 1.0f;

  // operands of one timestep, fetched one step ahead of their use
  struct Ops {
    ulonglong2 bq[4], cq[4];
    float dt[RPL], x[RPL];
  };
  auto load_ops = [&](Ops& o, const float* pB, const float* pC, const float* pX, const float* pD, int t) {
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      o.bq[m] = *reinterpret_cast<const ulonglong2*>(pB + t * N + 4 * LPR * m);
      o.cq[m] = *reinterpret_cast<const ulonglong2*>(pC + t * N + 4 * LPR * m);
    }
    if (RPL == 2) {
      const float2 d2 = *reinterpret_cast<const float2*>(pD + t * ROWS);
      const float2 x2 = *reinterpret_cast<const float2*>(pX + t * ROWS);
      o.dt[0] = d2.x; o.dt[RPL - 1] = d2.y; o.x[0] = x2.x; o.x[RPL - 1] = x2.y;
    } else {
#pragma unroll
      for (int r = 0; r < RPL; ++r) { o.dt[r] = pD[t * ROWS + r]; o.x[r] = pX[t * ROWS + r]; }
    }
  };

  // Reduce + D skip + gate + store of a block of four steps run one block LATE, interleaved with
  // the state updates of the next block, so the shuffle and MUFU latencies hide behind FMA work.
  // A lane finalises SPB = TPL / RPL steps (from step j*SPB of the block) of its RPL rows; their x
  // and z are captured in registers when the block is computed, so nothing depends on the tile.
  constexpr int SPB = TPL / RPL;
  float ypv[NV], fx[TPL], fz[TPL];
#pragma unroll
  for (int i = 0; i < NV; ++i) ypv[i] = 0.f;
#pragma unroll
  for (int i = 0; i < TPL; ++i) fx[i] = fz[i] = 0.f;
  float* fy = gY;
  int fvalid = 0;          // how many of the SPB owned steps exist
  auto finalize = [&]() {
#pragma unroll
    for (int r = 0; r < NR; ++r) {
      const int lane_bit = LPR >> (r + 1);
      const int cnt = (NV / 2) >> r;
      const bool hi = (j & lane_bit) != 0;
#pragma unroll
      for (int i = 0; i < cnt; ++i) {
        const float mine = hi ? ypv[i + cnt] : ypv[i];
        const float other = hi ? ypv[i] : ypv[i + cnt];
        ypv[i] = mine + __shfl_xor_sync(0xffffffffu, other, lane_bit);
      }
    }
#pragma unroll
    for (int sp = 0; sp < SPB; ++sp) {
      float y[RPL];
#pragma unroll
      for (int r = 0; r < RPL; ++r) {
        y[r] = fmaf(fx[sp * RPL + r], Dv[r], ypv[sp * RPL + r]);
        if (gate) {   // y * silu(z) = y * z / (1 + 2^(-z log2 e))
          const float zv = fz[sp * RPL + r];
          float sg;
          asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(sg) : "f"(1.0f + ex2_approx(-zv * LOG2E)));
          y[r] *= zv * sg;
        }
      }
      if (sp < fvalid) {
        if (RPL == 2) {
          *reinterpret_cast<float2*>(fy + sp * a.ldy) = make_float2(y[0], y[RPL - 1]);
        } else {
#pragma unroll
          for (int r = 0; r < RPL; ++r) fy[sp * a.ldy + r] = y[r];
        }
      }
    }
  };

  constexpr int NST = 3;   // tile stages: chunk c+2 is in flight while chunk c is consumed
  issue(0);
  issue(1);
  for (int c = 0; c < nchunks; ++c) {
    const int st = c % NST;
    const int64_t tc0 = (int64_t)c * TCH;
    const int tcn = (int)((L - tc0) < TCH ? (L - tc0) : TCH);
    cp_async_wait<1>();                   // every chunk but the newest has landed (for this thread)
    __syncthreads();                      // ... for every thread; and everyone is done with chunk c-1
    issue(c + 2);                         // refills the stage of chunk c-1
    const float* pB = sB(st) + 4 * j;
    const float* pC = sC(st) + 4 * j;
    const float* pX = sX(st) + rl0;
    const float* pD = sDt(st) + rl0;
    const float* pZ = sZ(st) + rl0;

    Ops cur;
    load_ops(cur, pB, pC, pX, pD, 0);
    Pre pre;
    auto mufu_phase = [&](const Ops& o, float (&r)[RPL], float (&e)[RPL], float (&rq)[RPL]) {
#pragma unroll
      for (int q = 0; q < RPL; ++q) {
        r[q] = ex2_approx(o.dt[q] * c_r);
        e[q] = ex2_approx(o.dt[q] * c_e);
        rq[q] = ex2_approx(o.dt[q] * c_q);
      }
    };
    auto pack_phase = [&](const Ops& o, const float (&r)[RPL], const float (&e)[RPL], const float (&rq)[RPL],
                          const float (&s_prev)[RPL], Pre& p) {
#pragma unroll
      for (int q = 0; q < RPL; ++q) {
        float u = o.x[q] * o.dt[q];
        if (fabsf(u) < 1e-12f) u = copysignf(1e-12f, u);
        float inv;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(u));
        const float er = e[q] * (s_prev[q] * inv);          // r^(4j+1) * u_{t-1} / u_t
        const float r2 = r[q] * r[q];
        p.Pa[q] = pack2(er, er * r[q]);
        p.Pb[q] = mul2(p.Pa[q], pack2(r2, r2));
        p.rq2[q] = pack2(rq[q], rq[q]);
        p.s[q] = u;
      }
    };
    if (STRUCT) {
      float r[RPL], e[RPL], rq[RPL];
      mufu_phase(cur, r, e, rq);
      pack_phase(cur, r, e, rq, s_carry, pre);
    }
#pragma unroll 4   // the whole 16-step chunk: no loop-carried register copies, no issue bubble at block ends (0.315 -> 0.292 ms)
    for (int g4 = 0; g4 < TCH; g4 += 4) {
      if (g4 >= tcn) break;
      float yp[NV];   // index RPL*i + r : step i, row r
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int t = g4 + i;
        Ops nxt;
        load_ops(nxt, pB, pC, pX, pD, t + 1 < TCH ? t + 1 : TCH - 1);
        if (STRUCT) {
          float r[RPL], e[RPL], rq[RPL];
          Pre npre;
          yp[RPL * i] = row_step_pre(H[0], pre.Pa[0], pre.Pb[0], pre.rq2[0], pre.s[0], cur.bq, cur.cq);
          mufu_phase(nxt, r, e, rq);
#pragma unroll
          for (int q = 1; q < RPL; ++q)
            yp[RPL * i + q] = row_step_pre(H[q], pre.Pa[q], pre.Pb[q], pre.rq2[q], pre.s[q], cur.bq, cur.cq);
#pragma unroll
          for (int q = 0; q < RPL; ++q) s_carry[q] = pre.s[q];
          pack_phase(nxt, r, e, rq, s_carry, npre);
          pre = npre;
        } else {
#pragma unroll
          for (int r = 0; r < RPL; ++r) yp[RPL * i + r] = row_step(H[r], cur.dt[r], cur.x[r], cur.bq, cur.cq);
        }
        cur = nxt;
      }
      // x and z of the values this lane will finalise one block from now
      float nfx[TPL], nfz[TPL];
      const int s0 = g4 + j * SPB;
#pragma unroll
      for (int sp = 0; sp < SPB; ++sp) {
        if (RPL == 2) {
          const float2 x2 = *reinterpret_cast<const float2*>(pX + (s0 + sp) * ROWS);
          const float2 z2 = gate ? *reinterpret_cast<const float2*>(pZ + (s0 + sp) * ROWS) : make_float2(0.f, 0.f);
          nfx[sp * RPL] = x2.x; nfx[sp * RPL + RPL - 1] = x2.y;
          nfz[sp * RPL] = z2.x; nfz[sp * RPL + RPL - 1] = z2.y;
        } else {
#pragma unroll
          for (int r = 0; r < RPL; ++r) {
            nfx[sp * RPL + r] = pX[(s0 + sp) * ROWS + r];
            nfz[sp * RPL + r] = gate ? pZ[(s0 + sp) * ROWS + r] : 0.f;
          }
        }
      }
      finalize();                          // the PREVIOUS block
#pragma unroll
      for (int i = 0; i < NV; ++i) ypv[i] = yp[i];
#pragma unroll
      for (int i = 0; i < TPL; ++i) { fx[i] = nfx[i]; fz[i] = nfz[i]; }
      fy = gY + (tc0 + s0) * a.ldy;
      fvalid = tcn - s0;
    }
  }
  // Programmatic launch of the next kernel only now: this grid is a single wave that runs for the whole
  // sequence (milliseconds at 600 s utterances), and CTAs of the next kernel that sit resident in
  // griddepcontrol.wait all that time cost this issue-bound kernel dearly (config 4: 124 ms per batch with the
  // trigger at the top of the kernel, 79 ms without programmatic launch at all).
  pdl_trigger();
  finalize();
}

// ------------------------------------------------------------------------------------------
// Row-packed recurrence kernel: the true recurrence for structured A and N = 64 (every shape the model runs).
//
// What was measured on scan_seq_kernel at batch 64 (ncu: profiles/scan_ncu.json; batch sweep: tools/scan_bench.py):
// every lane needs the 16 B and 16 C values of its states in registers each step, for only two rows — 4 KB per
// warp-step through the 128 B/clk shared-memory -> register path (41 wavefronts per warp-step, 69 % of the LSU data
// pipe); a third of the FMA-pipe time goes to scalar set-up arithmetic; and 384 CTAs over 148 SMs leave 3 CTAs on
// the critical SMs against 2.59 on average (0.20 ms at 2 CTAs per SM, 0.27 ms at 3: the time is a step function
// of the CTAs on the fullest SM).  This kernel changes all three:
//   * a packed fp32x2 register holds the SAME state of TWO ROWS (a row pair), not two states of one row.  B[n] and
//     C[n] then enter the FFMA2 as scalar-broadcast operands (SASS `.F32`, addend and multiplicand alike), so one
//     16-byte load of B feeds 2 * RP rows; with RP = 2 row pairs per lane (4 rows, 64 state registers) the B / C
//     traffic per row halves (10.5 LDS.128 per 32-row warp-step);
//   * all per-row set-up (exponent arguments, u = x dt, the ratio of consecutive scales, the power seeds) runs as
//     packed operations on the pair;
//   * the time axis is cut at chunk boundaries and dealt out evenly: the grid is a fixed number of slots
//     (resident CTAs), slot s owns the range [s T / S, (s + 1) T / S) of the chunk sequence of all chains laid end
//     to end (a chain = the rows of one CTA x the whole utterance).  A slot first runs the pieces that start a chain
//     (no dependency), last the tail of the chain its range begins in, which continues from the state the previous
//     slot published (state + carried scale through global memory, one flag per slot).  The split changes no
//     arithmetic: a row sees exactly the operation sequence of the unsplit recurrence, whatever the CTA shape.
// Everything else follows scan_seq_kernel: cp.async tiles in natural layout three stages deep, operands and set-up
// one step ahead, state carried divided by the input, transpose-reduce of four steps across the four lanes of a
// row group one block late, D skip + silu(z) gate + 16-byte store by the lane that ends up with a finished value.
//
// What it bought, and what bounds it now (same box, 64 / 128 / 512 x 751 x 384): 0.252 / 0.420 / 1.57 ms against
// 0.268 / 0.498 / 1.64 ms.  184.75 instructions per 32-row warp-step (116 packed; scan_seq_kernel: 124.5 per 16
// rows, 48 packed), LSU data pipe 49 %, FMA pipe 62 %, XU 39 % at two warps per sub-partition: no pipe saturates.
// A fit over both kernels prices a packed instruction at ~2.8 clocks and any other at ~1.2, i.e. the three packed
// operations per state and step (47 per 16 rows: ~130 clocks) are two thirds of the time, and a warp alone on its
// sub-partition issues in 45 % of the cycles (37 % fixed-latency waits of the in-order pipe).  A third CTA per SM
// (168 registers, two tile stages) and a fully unrolled 16-step body (48 KB of code: instruction-cache misses were
// the top stall) were both slower.  At batch 64 the floor is the chain itself: 751 sequential steps at the pace
// of a sub-partition that two warps share.
// ------------------------------------------------------------------------------------------
struct SplitArgs {
  u64* state = nullptr;           // per slot: THREADS * (RP * 17) packed values (RP * 16 states + RP carried scales)
  unsigned int* flags = nullptr;  // per slot: launch epoch once the slot's state is published
  unsigned int epoch = 0;
  int n_slots = 0;
};

__device__ __forceinline__ u64 shfl_xor2(u64 v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
__device__ __forceinline__ u64 bcast2(float v) { return pack2(v, v); }
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

template <int RP, int WARPS, int OCC>   // OCC: CTAs per SM the register budget is cut for
__global__ void __launch_bounds__(WARPS * 32, OCC) scan_rp_kernel(ScanArgs a, SplitArgs sa) {
  pdl_wait();
  constexpr int N = 64, G = 8, R = 2 * RP;      // 4 lanes per row group, G groups per warp, R rows per lane
  constexpr int ROWS = WARPS * G * R;
  constexpr int THREADS = WARPS * 32;
  constexpr int LDR = ROWS + 8;                 // row stride of the x / dt / z tiles: the finalising lanes of a group
                                                // read four different timesteps, 8 floats of padding keep them apart
  constexpr int NF = N / 4, RF = ROWS / 4;
  constexpr int STAGE_FLOATS = TCH * (2 * N + 3 * LDR);
  constexpr int NST = 3;                        // tile stages: chunk c in use, c + 1 landed, c + 2 in flight
  constexpr int NV = 4 * RP;                    // packed partials per lane per block of four steps
  constexpr int SW = RP * 17;                   // packed values per thread in a published state

  extern __shared__ __align__(16) float scan_smem[];
  auto sB = [&](int st) { return scan_smem + st * STAGE_FLOATS; };
  auto sC = [&](int st) { return scan_smem + st * STAGE_FLOATS + TCH * N; };
  auto sX = [&](int st) { return scan_smem + st * STAGE_FLOATS + 2 * TCH * N; };
  auto sDt = [&](int st) { return scan_smem + st * STAGE_FLOATS + 2 * TCH * N + TCH * LDR; };
  auto sZ = [&](int st) { return scan_smem + st * STAGE_FLOATS + 2 * TCH * N + 2 * TCH * LDR; };

  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, j = lane & 3;
  const int rl0 = (warp * G + g) * R;
  const int64_t L = a.L;
  const bool gate = a.z != nullptr;
  const int tiles = a.Di / ROWS;
  const int64_t cpc = (L + TCH - 1) / TCH;                  // chunks per chain
  const int64_t n_chains = a.B * tiles;

  // this slot's range of the chunk sequence of all chains laid end to end
  int64_t f0, f1;
  if (sa.n_slots > 0) {
    const int64_t total = n_chains * cpc;
    f0 = total * blockIdx.x / sa.n_slots;
    f1 = total * (blockIdx.x + 1) / sa.n_slots;
  } else {
    f0 = (int64_t)blockIdx.x * cpc;
    f1 = f0 + cpc;
  }
  if (f1 <= f0) {
    pdl_trigger();
    return;
  }
  const int64_t c_first = f0 / cpc, c_last = (f1 - 1) / cpc;

  const u64 CR = bcast2(-LOG2E);                            // r  = exp(-dt)
  const u64 CE = bcast2(-LOG2E * (float)(4 * j + 1));       // e  = r^(4j+1)
  const u64 CQ = bcast2(-LOG2E * 16.0f);                    // rq = r^16: states 4 (j + 4 m) + i, m = 0..3

  // pieces in descending chain order: the ones that start a chain first, the dependent tail last
  for (int64_t chain = c_last; chain >= c_first; --chain) {
    const int cb = (int)((f0 > chain * cpc ? f0 : chain * cpc) - chain * cpc);
    const int ce = (int)((f1 < (chain + 1) * cpc ? f1 : (chain + 1) * cpc) - chain * cpc);
    const bool load_state = cb > 0, save_state = ce < cpc;
    const bool last_piece = chain == c_first;
    const int64_t b = chain / tiles;
    const int d0 = (int)(chain % tiles) * ROWS;

    u64 DV[RP];
#pragma unroll
    for (int p = 0; p < RP; ++p)
      DV[p] = a.D ? pack2(__ldg(a.D + d0 + rl0 + 2 * p), __ldg(a.D + d0 + rl0 + 2 * p + 1)) : 0ull;

    const float* gB = a.Bm + b * L * a.ldb;
    const float* gC = a.Cm + b * L * a.ldc;
    const float* gX = a.x + b * L * a.ldx + d0;
    const float* gDt = a.dt + b * L * a.lddt + d0;
    const float* gZ = gate ? a.z + b * L * a.ldz + d0 : nullptr;
    float* gY = a.y + b * L * a.ldy + d0 + rl0;

    // Tile loads.  Thread tid moves, per chunk, the float4 pieces (t = tb + TSB i, f = tid % NF) of B and C and
    // (t = tx + TSX i, f = tid % RF) of x / dt / z: fixed per-thread offsets, so a chunk costs one pointer advance
    // per array and no index arithmetic (the first version recomputed every address from tid and re-read the
    // strides from the constant bank: 345 instructions per chunk, 18 % of a lone warp's time).
    constexpr int TSB = THREADS / NF, TSX = THREADS / RF;      // timesteps between a thread's pieces
    static_assert(THREADS % NF == 0 && THREADS % RF == 0 && TCH % TSB == 0 && TCH % TSX == 0, "tile shape");
    const int tb = tid / NF, fb = tid % NF, tx = tid / RF, fx = tid % RF;
    const float* qB = gB + ((int64_t)cb * TCH + tb) * a.ldb + 4 * fb;
    const float* qC = gC + ((int64_t)cb * TCH + tb) * a.ldc + 4 * fb;
    const float* qX = gX + ((int64_t)cb * TCH + tx) * a.ldx + 4 * fx;
    const float* qD = gDt + ((int64_t)cb * TCH + tx) * a.lddt + 4 * fx;
    const float* qZ = gate ? gZ + ((int64_t)cb * TCH + tx) * a.ldz + 4 * fx : nullptr;
    const int oB = tb * N + 4 * fb, oX = tx * LDR + 4 * fx;     // offsets inside a stage
    int c_issue = cb;                                            // next chunk to be requested
    auto issue = [&]() {               // always commits a group (an empty one past the piece's last chunk)
      const int c = c_issue++;
      if (c < ce) {
        const int st = (c - cb) % NST;
        float* dB = sB(st) + oB; float* dC = sC(st) + oB;
        float* dX = sX(st) + oX; float* dD = sDt(st) + oX; float* dZ = sZ(st) + oX;
        const int64_t left = L - (int64_t)c * TCH;               // timesteps this chunk holds
        if (left >= TCH) {
#pragma unroll
          for (int i = 0; i < TCH / TSB; ++i) {
            cp_async16(dB + i * TSB * N, qB + (int64_t)i * TSB * a.ldb);
            cp_async16(dC + i * TSB * N, qC + (int64_t)i * TSB * a.ldc);
          }
#pragma unroll
          for (int i = 0; i < TCH / TSX; ++i) {
            cp_async16(dX + i * TSX * LDR, qX + (int64_t)i * TSX * a.ldx);
            cp_async16(dD + i * TSX * LDR, qD + (int64_t)i * TSX * a.lddt);
            if (gate) cp_async16(dZ + i * TSX * LDR, qZ + (int64_t)i * TSX * a.ldz);
          }
        } else {                                                 // the last chunk of a chain
#pragma unroll
          for (int i = 0; i < TCH / TSB; ++i)
            if (tb + i * TSB < left) {
              cp_async16(dB + i * TSB * N, qB + (int64_t)i * TSB * a.ldb);
              cp_async16(dC + i * TSB * N, qC + (int64_t)i * TSB * a.ldc);
            }
#pragma unroll
          for (int i = 0; i < TCH / TSX; ++i)
            if (tx + i * TSX < left) {
              cp_async16(dX + i * TSX * LDR, qX + (int64_t)i * TSX * a.ldx);
              cp_async16(dD + i * TSX * LDR, qD + (int64_t)i * TSX * a.lddt);
              if (gate) cp_async16(dZ + i * TSX * LDR, qZ + (int64_t)i * TSX * a.ldz);
            }
        }
        qB += (int64_t)TCH * a.ldb; qC += (int64_t)TCH * a.ldc;
        qX += (int64_t)TCH * a.ldx; qD += (int64_t)TCH * a.lddt;
        if (gate) qZ += (int64_t)TCH * a.ldz;
      }
      cp_async_commit();
    };
#pragma unroll
    for (int i = 0; i < NST - 1; ++i) issue();                // the tiles travel while the state is fetched

    // ---- state: zero at the start of a chain, else what the previous slot published
    u64 H[RP][16];
    u64 s_carry[RP];
    if (load_state) {
      if (tid == 0) {
        const volatile unsigned int* fl = sa.flags + (blockIdx.x - 1);
        const unsigned long long t0 = global_ns();
        while (*fl != sa.epoch) {
          __nanosleep(100);
          if (global_ns() - t0 > 4000000000ull) __trap();     // 4 s: a lost hand-over must not hang the device
        }
        __threadfence();
      }
      __syncthreads();
      const u64* st = sa.state + (size_t)(blockIdx.x - 1) * THREADS * SW + tid;
#pragma unroll
      for (int p = 0; p < RP; ++p) {
#pragma unroll
        for (int k = 0; k < 16; ++k) H[p][k] = __ldcg(st + (size_t)(p * 16 + k) * THREADS);
        s_carry[p] = __ldcg(st + (size_t)(RP * 16 + p) * THREADS);
      }
    } else {
#pragma unroll
      for (int p = 0; p < RP; ++p) {
#pragma unroll
        for (int k = 0; k < 16; ++k) H[p][k] = 0ull;
        s_carry[p] = bcast2(1.0f);
      }
    }

    // set-up of one step for one row pair, from its dt and x (packed over the two rows)
    struct Pre {
      u64 ER[RP], R1[RP], R2[RP], RQ[RP], S[RP];
    };
    struct Raw {       // MUFU results of a step's set-up, before they are combined
      float r[R], e[R], q[R], u[R], inv[R];
    };
    auto load_dx = [&](u64 (&DT)[RP], u64 (&X)[RP], const float* pD, const float* pX, int t) {
      if (RP == 2) {
        const ulonglong2 d = *reinterpret_cast<const ulonglong2*>(pD + t * LDR);
        const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(pX + t * LDR);
        DT[0] = d.x; DT[RP - 1] = d.y; X[0] = x.x; X[RP - 1] = x.y;
      } else {
        DT[0] = *reinterpret_cast<const u64*>(pD + t * LDR);
        X[0] = *reinterpret_cast<const u64*>(pX + t * LDR);
      }
    };
    auto mufu_phase = [&](const u64 (&DT)[RP], const u64 (&X)[RP], Raw& w) {
#pragma unroll
      for (int p = 0; p < RP; ++p) {
        float a0, a1;
        unpack2(mul2(DT[p], CR), a0, a1);
        w.r[2 * p] = ex2_approx(a0); w.r[2 * p + 1] = ex2_approx(a1);
        unpack2(mul2(DT[p], CE), a0, a1);
        w.e[2 * p] = ex2_approx(a0); w.e[2 * p + 1] = ex2_approx(a1);
        unpack2(mul2(DT[p], CQ), a0, a1);
        w.q[2 * p] = ex2_approx(a0); w.q[2 * p + 1] = ex2_approx(a1);
        unpack2(mul2(X[p], DT[p]), a0, a1);
        if (fabsf(a0) < 1e-12f) a0 = copysignf(1e-12f, a0);
        if (fabsf(a1) < 1e-12f) a1 = copysignf(1e-12f, a1);
        w.u[2 * p] = a0; w.u[2 * p + 1] = a1;
        w.inv[2 * p] = rcp_approx(a0); w.inv[2 * p + 1] = rcp_approx(a1);
      }
    };
    auto pack_phase = [&](const Raw& w, const u64 (&s_prev)[RP], Pre& o) {
#pragma unroll
      for (int p = 0; p < RP; ++p) {
        const u64 ratio = mul2(s_prev[p], pack2(w.inv[2 * p], w.inv[2 * p + 1]));     // u_{t-1} / u_t
        o.ER[p] = mul2(pack2(w.e[2 * p], w.e[2 * p + 1]), ratio);                     // r^(4j+1) u_{t-1} / u_t
        o.R1[p] = pack2(w.r[2 * p], w.r[2 * p + 1]);
        o.R2[p] = mul2(o.R1[p], o.R1[p]);
        o.RQ[p] = pack2(w.q[2 * p], w.q[2 * p + 1]);
        o.S[p] = pack2(w.u[2 * p], w.u[2 * p + 1]);
      }
    };

    // finalisation (one block of four steps late): see scan_seq_kernel
    u64 ypv[NV], FX[RP], FZ[RP];
#pragma unroll
    for (int i = 0; i < NV; ++i) ypv[i] = 0ull;
#pragma unroll
    for (int p = 0; p < RP; ++p) FX[p] = FZ[p] = 0ull;
    float* fy = gY;
    bool fvalid = false;
    auto finalize = [&]() {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int lane_bit = 2 >> r;
        const int cnt = (NV / 2) >> r;
        const bool hi = (j & lane_bit) != 0;
#pragma unroll
        for (int i = 0; i < cnt; ++i) {
          const u64 mine = hi ? ypv[i + cnt] : ypv[i];
          const u64 other = hi ? ypv[i] : ypv[i + cnt];
          ypv[i] = add2(mine, shfl_xor2(other, lane_bit));
        }
      }
      float out[R];
#pragma unroll
      for (int p = 0; p < RP; ++p) {
        u64 y = fma2(FX[p], DV[p], ypv[p]);
        if (gate) {          // y * silu(z) = y * z / (1 + 2^(-z log2 e))
          float e0, e1;
          unpack2(mul2(FZ[p], CR), e0, e1);
          const u64 sg = pack2(rcp_approx(1.0f + ex2_approx(e0)), rcp_approx(1.0f + ex2_approx(e1)));
          y = mul2(y, mul2(FZ[p], sg));
        }
        unpack2(y, out[2 * p], out[2 * p + 1]);
      }
      if (fvalid) {
        if (RP == 2) *reinterpret_cast<float4*>(fy) = make_float4(out[0], out[1], out[R - 2], out[R - 1]);
        else *reinterpret_cast<float2*>(fy) = make_float2(out[0], out[1]);
      }
    };

    // One barrier per chunk, at the start of its LAST block of four steps: by then every thread's part of chunk
    // c + 1 has landed (wait_group), after it that chunk is visible to all, and every thread has left chunk c - 1,
    // whose stage takes the request for chunk c + 2.  Placed there — not at the top of a chunk — the set-up
    // of step 0 of the next chunk runs behind the last step of this one like any other step's, instead of as a
    // serial MUFU chain at every chunk start.
    cp_async_wait<NST - 2>();
    __syncthreads();                        // the piece's first chunk is in place
    Pre pre;
    {
      u64 DT[RP], X[RP];
      Raw w;
      load_dx(DT, X, sDt(0) + rl0, sX(0) + rl0, 0);
      mufu_phase(DT, X, w);
      pack_phase(w, s_carry, pre);
    }
    for (int c = cb; c < ce; ++c) {
      const int st = (c - cb) % NST, stn = (c + 1 - cb) % NST;
      const int64_t tc0 = (int64_t)c * TCH;
      const int tcn = (int)((L - tc0) < TCH ? (L - tc0) : TCH);
      if (last_piece && c + 1 == ce) pdl_trigger();   // single-wave long runner: let the next kernel queue up late
      const float* pB = sB(st) + 4 * j;
      const float* pC = sC(st) + 4 * j;
      const float* pX = sX(st) + rl0;
      const float* pD = sDt(st) + rl0;
      const float* pZ = sZ(st) + rl0;
      // one block of four steps is the loop body (not the whole chunk as in scan_seq_kernel): 200 instructions per
      // step for RP = 2, and a 16-step body (48 KB of code) ran out of instruction cache ("no instruction" was the
      // top stall reason in the first capture of this kernel)
#pragma unroll 1
      for (int g4 = 0; g4 < TCH; g4 += 4) {
        if (g4 >= tcn) break;
        const bool last_block = g4 + 4 == TCH;
        if (last_block) {
          cp_async_wait<0>();                 // chunk c + 1 (the only request in flight) has landed
          __syncthreads();
          issue();                            // chunk c + 2, into the stage chunk c - 1 has just left
        }
        // dt / x of the step after this block's last: row 0 of the next chunk's stage at the end of a chunk
        const float* pDl = last_block ? sDt(stn) + rl0 : pD + (g4 + 4) * LDR;
        const float* pXl = last_block ? sX(stn) + rl0 : pX + (g4 + 4) * LDR;
        u64 yp[NV];      // index RP * i + p : step i of the block, row pair p
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int t = g4 + i;
          u64 DTn[RP], Xn[RP];
          Raw w;
          Pre npre;
          if (i < 3) load_dx(DTn, Xn, pD, pX, t + 1);
          else load_dx(DTn, Xn, pDl, pXl, 0);
          u64 P[RP][4], acc[RP][2];
#pragma unroll
          for (int p = 0; p < RP; ++p) {
            P[p][0] = pre.ER[p];
            P[p][1] = mul2(pre.ER[p], pre.R1[p]);
            P[p][2] = mul2(pre.ER[p], pre.R2[p]);
            P[p][3] = mul2(P[p][1], pre.R2[p]);
          }
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            const float4 bq = *reinterpret_cast<const float4*>(pB + t * N + 16 * m);
            const float4 cq = *reinterpret_cast<const float4*>(pC + t * N + 16 * m);
            const float bv[4] = {bq.x, bq.y, bq.z, bq.w};
            const float cv[4] = {cq.x, cq.y, cq.z, cq.w};
#pragma unroll
            for (int p = 0; p < RP; ++p) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                u64& h = H[p][4 * m + q];
                h = fma2(P[p][q], h, bcast2(bv[q]));
                if (m == 0 && q < 2) acc[p][q] = mul2(h, bcast2(cv[q]));
                else acc[p][q & 1] = fma2(h, bcast2(cv[q]), acc[p][q & 1]);
                if (m < 3) P[p][q] = mul2(P[p][q], pre.RQ[p]);
              }
            }
            if (m == 0) mufu_phase(DTn, Xn, w);       // the MUFU results of step t+1 mature behind the FMA work
          }
#pragma unroll
          for (int p = 0; p < RP; ++p) {
            yp[RP * i + p] = mul2(add2(acc[p][0], acc[p][1]), pre.S[p]);
            s_carry[p] = pre.S[p];
          }
          pack_phase(w, s_carry, npre);
          pre = npre;
        }
        // x and z of the step this lane will finalise one block from now
        u64 nFX[RP], nFZ[RP];
        const int s0 = g4 + j;
        if (RP == 2) {
          const ulonglong2 x2 = *reinterpret_cast<const ulonglong2*>(pX + s0 * LDR);
          nFX[0] = x2.x; nFX[RP - 1] = x2.y;
          if (gate) {
            const ulonglong2 z2 = *reinterpret_cast<const ulonglong2*>(pZ + s0 * LDR);
            nFZ[0] = z2.x; nFZ[RP - 1] = z2.y;
          } else {
            nFZ[0] = nFZ[RP - 1] = 0ull;
          }
        } else {
          nFX[0] = *reinterpret_cast<const u64*>(pX + s0 * LDR);
          nFZ[0] = gate ? *reinterpret_cast<const u64*>(pZ + s0 * LDR) : 0ull;
        }
        finalize();                          // the PREVIOUS block
#pragma unroll
        for (int i = 0; i < NV; ++i) ypv[i] = yp[i];
#pragma unroll
        for (int p = 0; p < RP; ++p) { FX[p] = nFX[p]; FZ[p] = nFZ[p]; }
        fy = gY + (tc0 + s0) * a.ldy;
        fvalid = s0 < tcn;
      }
    }
    finalize();
    cp_async_wait<0>();

    if (save_state) {       // hand the chain over to the next slot
      u64* st = sa.state + (size_t)blockIdx.x * THREADS * SW + tid;
#pragma unroll
      for (int p = 0; p < RP; ++p) {
#pragma unroll
        for (int k = 0; k < 16; ++k) __stcg(st + (size_t)(p * 16 + k) * THREADS, H[p][k]);
        __stcg(st + (size_t)(RP * 16 + p) * THREADS, s_carry[p]);
      }
      __threadfence();
      __syncthreads();
      if (tid == 0) *reinterpret_cast<volatile unsigned int*>(sa.flags + blockIdx.x) = sa.epoch;
    } else {
      __syncthreads();      // the next piece re-uses the tile stages
    }
  }
}

// Row-packed kernel, two shapes with identical per-row arithmetic (a row's result does not depend on which one ran,
// nor on where the time axis was cut): 128-row CTAs (two row pairs per lane) when that still gives every SM a
// chain, 64-row CTAs (one pair per lane) for smaller batches.
constexpr int RP_WARPS = 4;
template <int RP, int OCC = 3>
struct RpCfg {
  static constexpr int ROWS = RP_WARPS * 8 * 2 * RP;
  static constexpr int THREADS = RP_WARPS * 32;
  static constexpr size_t SMEM = (size_t)3 * TCH * (2 * 64 + 3 * (ROWS + 8)) * sizeof(float);
  static constexpr size_t STATE_BYTES = (size_t)THREADS * RP * 17 * sizeof(unsigned long long);   // per slot
};
constexpr int RP_MAX_SLOTS = 1024;
constexpr size_t RP_SCRATCH_BYTES = 4096 + (size_t)RP_MAX_SLOTS * RpCfg<2>::STATE_BYTES;

// Hand-over scratch of the time split: one per (device, stream), made on first use and kept.  Launches on one
// stream are serialised, so they can share it; the flags are zeroed once and every launch uses a new epoch.
// (A captured CUDA graph would replay a stale epoch: launch_selective_scan is not graph-capturable when it splits.)
struct RpScratch {
  void* mem = nullptr;
  unsigned int epoch = 0;
};
cudaError_t rp_scratch(cudaStream_t s, RpScratch** out) {
  static std::mutex mu;
  static std::map<std::pair<int, cudaStream_t>, RpScratch> cache;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  RpScratch& sc = cache[std::make_pair(dev, s)];
  if (!sc.mem) {
    e = cudaMalloc(&sc.mem, RP_SCRATCH_BYTES);
    if (e != cudaSuccess) return e;
    e = cudaMemset(sc.mem, 0, 4096);
    if (e != cudaSuccess) return e;
  }
  *out = &sc;
  return cudaSuccess;
}

// true when the row-packed kernel takes this problem: true recurrence, structured A, N = 64, whole CTAs of rows,
// 16-byte aligned rows
bool rp_takes(const ScanArgs& a) {
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  if (a.parallel_quirk || !a.structured_a || a.N != 64 || a.Di % RpCfg<1>::ROWS != 0) return false;
  if ((a.ldx & 3) || (a.lddt & 3) || (a.ldy & 3) || (a.ldb & 3) || (a.ldc & 3)) return false;
  if (!al16(a.x) || !al16(a.dt) || !al16(a.y) || !al16(a.Bm) || !al16(a.Cm)) return false;
  if (a.z && ((a.ldz & 3) || !al16(a.z))) return false;
  return true;
}

// where each launch site records what it launched (scan_last_variant)
thread_local ScanVariant scan_variant_rec;

template <int RP, int OCC>
cudaError_t launch_rp_cfg(const ScanArgs& a, int sms, int split_ov, cudaStream_t s) {
  using C = RpCfg<RP, OCC>;
  auto kernel = scan_rp_kernel<RP, RP_WARPS, OCC>;
  // A split launch asks for at least SPLIT_SMEM bytes of shared memory, more than a third of an SM's: never more
  // than two CTAs per SM.  The slots are dealt two per SM; under programmatic launch the CTAs arrive while the
  // previous kernel drains, and with room for three the SMs that free first took three slots and left others with
  // one (step 5.47 -> 6.02 ms before this cap).
  constexpr size_t SPLIT_SMEM = C::SMEM > 78 * 1024 ? C::SMEM : 78 * 1024;
  static int occ = -1;
  cudaError_t e = cudaSuccess;
  if (occ < 0) {
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SPLIT_SMEM);
    if (e != cudaSuccess) return e;
    int n = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, C::THREADS, C::SMEM);
    if (e != cudaSuccess) return e;
    occ = n;
  }
  const int64_t n_chains = a.B * (a.Di / C::ROWS);
  const int64_t total = n_chains * ((a.L + TCH - 1) / TCH);
  SplitArgs sa;
  unsigned grid = (unsigned)n_chains;
  size_t smem = C::SMEM;
  // Time split into two slots per SM, when there are more chains than that and they do not divide evenly.  What a
  // split can and cannot do (tools/scan_variants.sh, batch 64 x 751): a chain stays 751 sequential steps whose pace
  // is set by how many warps share its sub-partition, so cutting chains that already fit the resident slots only
  // adds co-residents and slows every chain (444 slots: 0.264 ms; 296: 0.252; unsplit 384 CTAs: 0.269); the gain
  // is in evening out MORE chains than slots (1.3 chains per slot instead of 3 CTAs on some SMs and 2 on others).
  // A slot may wait for its predecessor only, which the hardware dispatched before it (CTAs are dealt out in index
  // order).
  int64_t slots = (int64_t)(occ < 2 ? occ : 2) * sms;
  if (slots > RP_MAX_SLOTS) slots = RP_MAX_SLOTS;
  if (slots > total) slots = total;
  if (split_ov > 0 && split_ov <= (int64_t)occ * sms && split_ov <= RP_MAX_SLOTS) slots = split_ov;
  bool split = occ > 0 && n_chains > slots && slots >= 1 && n_chains % slots != 0;
  if (split_ov < 0) split = false;
  if (split) {
    RpScratch* sc = nullptr;
    e = rp_scratch(s, &sc);
    if (e != cudaSuccess) return e;
    sa.n_slots = (int)slots;
    sa.flags = reinterpret_cast<unsigned int*>(sc->mem);
    sa.state = reinterpret_cast<u64*>(reinterpret_cast<char*>(sc->mem) + 4096);
    if (++sc->epoch == 0) ++sc->epoch;              // 0 is what the zeroed flags hold
    sa.epoch = sc->epoch;
    grid = (unsigned)slots;
    smem = SPLIT_SMEM;
  }
  scan_variant_rec = {3, RP, RP_WARPS, OCC, 1, sa.n_slots};
  scan_last_variant = &scan_variant_rec;
  return launch_k(kernel, dim3(grid), dim3(C::THREADS), smem, s, a, sa);
}

cudaError_t launch_rp(const ScanArgs& a, const ScanOverride& ov, cudaStream_t s) {
  const int sms = a.num_sms > 0 ? a.num_sms : 148;
  // 128-row CTAs once they fill two slots per SM (batch 128: 0.42 ms against 0.47 for 64-row CTAs and 0.50 for
  // scan_seq_kernel); below that the 64-row shape keeps more chains in flight (batch 64: 0.252 against 0.308)
  const bool wide = a.Di % RpCfg<2>::ROWS == 0 && (ov.rp ? ov.rp == 2 : a.B * (a.Di / RpCfg<2>::ROWS) >= 2 * sms);
  if (wide) return launch_rp_cfg<2, 2>(a, sms, ov.split, s);
  return launch_rp_cfg<1, 3>(a, sms, ov.split, s);
}

template <int LPR, int WARPS, int RPL>
cudaError_t launch_seq(const ScanArgs& a, cudaStream_t s) {
  constexpr int N = LPR * 16;
  constexpr int ROWS = WARPS * (32 / LPR) * RPL;
  constexpr size_t SMEM = (size_t)3 * TCH * (2 * N + 3 * ROWS) * sizeof(float);
  dim3 grid((unsigned)(a.Di / ROWS), (unsigned)a.B);
  cudaError_t e = cudaSuccess;
  auto go = [&](auto kernel, bool st) {
    if (SMEM > 48 * 1024) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM);
    if (e != cudaSuccess) return;
    scan_variant_rec = {2, LPR, WARPS, RPL, st ? 1 : 0, 0};
    scan_last_variant = &scan_variant_rec;
    e = launch_k(kernel, grid, dim3(WARPS * 32), SMEM, s, a);
  };
  if (a.structured_a) go(scan_seq_kernel<LPR, WARPS, RPL, true>, true);
  else go(scan_seq_kernel<LPR, WARPS, RPL, false>, false);
  return e;
}

// CTA shape of scan_seq_kernel: two rows per lane, four warps of them if that is at most 128 rows and divides Di, else
// a 64-row CTA (Di is a multiple of 64: include/vasr.h).  Only those two shapes are compiled.
template <int LPR>
cudaError_t launch_recurrence(const ScanArgs& a, cudaStream_t s) {
  constexpr int RW = 2 * 32 / LPR;                      // rows per warp
  constexpr int W_WIDE = 128 / RW < 4 ? 128 / RW : 4;   // warps of the wider CTA
  constexpr int W_64 = 64 / RW;                         // warps of a 64-row CTA
  // cp.async moves 16-byte pieces: every row start must be 16-byte aligned
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  if ((a.ldx & 3) || (a.lddt & 3) || (a.ldy & 1) || !al16(a.x) || !al16(a.dt) || (a.z && ((a.ldz & 3) || !al16(a.z))) ||
      (reinterpret_cast<uintptr_t>(a.y) & 7))
    return cudaErrorInvalidValue;
  // four warps = one warp of the CTA per SM sub-partition: the warps of a CTA then advance at the same rate and the
  // per-chunk barrier costs nothing (measured 0.320 ms vs 0.356 ms with three)
  if (a.Di % (W_WIDE * RW) == 0) return launch_seq<LPR, W_WIDE, 2>(a, s);
  if constexpr (W_64 != W_WIDE) {
    if (a.Di % 64 == 0) return launch_seq<LPR, W_64, 2>(a, s);
  }
  return cudaErrorInvalidValue;
}

template <int LPR8>   // LPR8 = N / 8: lanes per row of the quirk kernel
cudaError_t launch_lpr(const ScanArgs& a, cudaStream_t s) {
  if (!a.parallel_quirk) return launch_recurrence<LPR8 / 2>(a, s);
  constexpr int ROWS = SCAN_THREADS / LPR8;
  if (a.Di % ROWS != 0) return cudaErrorInvalidValue;
  dim3 grid((unsigned)(a.Di / ROWS), (unsigned)a.B);
  scan_variant_rec = {1, LPR8, 0, 0, a.structured_a ? 1 : 0, 0};
  scan_last_variant = &scan_variant_rec;
  if (a.structured_a) return launch_k(scan_quirk_kernel<LPR8, true>, grid, dim3(SCAN_THREADS), 0, s, a);
  return launch_k(scan_quirk_kernel<LPR8, false>, grid, dim3(SCAN_THREADS), 0, s, a);
}

// VASR_SCAN_OLD=1: scan_seq_kernel for every shape; VASR_SCAN_RP=1 / 2: that CTA shape of scan_rp_kernel;
// VASR_SCAN_SPLIT=0: never split, n > 0: n slots.  (Read in the debug build only, common.cuh.)
ScanOverride env_override() {
  ScanOverride o;
  o.rp = debug_env_int("VASR_SCAN_OLD", 0) ? -1 : debug_env_int("VASR_SCAN_RP", 0);
  const int sp = debug_env_int("VASR_SCAN_SPLIT", -1);
  o.split = sp == 0 ? -1 : (sp > 0 ? sp : 0);
  return o;
}

}  // namespace

thread_local const ScanVariant* scan_last_variant = nullptr;

cudaError_t launch_selective_scan(const ScanArgs& a, cudaStream_t s, int64_t* launches, const ScanOverride* ov) {
  if (a.B <= 0 || a.L <= 0) return cudaSuccess;
  if (a.B > 65535 || a.L >= (1LL << (NLEV - 2))) return cudaErrorInvalidValue;
  if ((a.ldb & 3) || (a.ldc & 3) || (reinterpret_cast<uintptr_t>(a.Bm) & 15) ||
      (reinterpret_cast<uintptr_t>(a.Cm) & 15))
    return cudaErrorInvalidValue;
  static const ScanOverride env_ov = env_override();
  const ScanOverride& o = ov ? *ov : env_ov;
  cudaError_t e;
  const bool rp = rp_takes(a);
  if (ov && ov->rp > 0 && (!rp || (ov->rp == 2 && a.Di % RpCfg<2>::ROWS != 0)))   // a forced shape that does not fit
    return cudaErrorInvalidValue;
  if (rp && o.rp >= 0) {
    e = launch_rp(a, o, s);
    if (launches && e == cudaSuccess) ++*launches;
    return e;
  }
  switch (a.N) {
    case 64: e = launch_lpr<8>(a, s); break;
    case 32: e = launch_lpr<4>(a, s); break;
    case 16: e = launch_lpr<2>(a, s); break;
    default: return cudaErrorInvalidValue;
  }
  if (launches && e == cudaSuccess) ++*launches;
  return e;
}

}  // namespace vasr
