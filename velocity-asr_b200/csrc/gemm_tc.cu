// gemm_tc.cu — tensor-core projection kernel for sm_100a: C = epi(A · Wᵀ) with fp32-grade accuracy.
//
// tcgen05.mma (kind::tf32) issued by one thread; the weight operand is staged in shared memory
// by TMA (128-byte swizzle), the activation operand is fed from TENSOR MEMORY, accumulators live
// in TMEM and are read back with tcgen05.ld for a fused, coalesced epilogue.
//
// Accuracy.  One TF32 pass carries ~1e-3 relative error, which flips ~0.3 % of the CTC argmaxes
// (SURVEY.md section 7.3c).  Each fp32 operand is therefore split into hi + lo, both TF32 values
// (hi = rna_tf32(x), lo = rna_tf32(x - hi); round-to-nearest keeps the residual error unbiased, which
// matters for the 400-term DFT rows), and every k-step issues three MMAs,
// A_lo·W_hi + A_hi·W_lo + A_hi·W_hi, accumulated in fp32 in TMEM (error ~2^-22 per product).
//
// Where the split happens (round-1 ncu: the first version split both tiles in shared memory and was
// bound by shared-memory bandwidth — TMA write + converter read/write + 3x MMA operand reads):
//   * weights are split ONCE (launch_split_tf32, cached per weight matrix by the engine) and TMA
//     brings W_hi and W_lo tiles straight from L2;
//   * the activation tile arrives as raw fp32; four converter warps read it once (one row per
//     thread = one TMEM lane), split it in registers and tcgen05.st the hi and lo halves into TMEM,
//     from where the MMA reads its A operand.  Shared memory then carries only the TMA writes, one
//     read of A and the MMA reads of W.
//
// Structure (persistent, one CTA per SM, 14 warps):
//   warp 0      TMA producer      : A (128 x 32 fp32), W_hi and W_lo (128 x 32) per stage, 4 stages
//   warp 1      MMA issuer        : 12 tcgen05.mma per stage; tcgen05.commit frees the stage
//   warps 2-5   converters        : smem A row -> hi/lo -> TMEM (64 columns per stage)
//   warps 6-13  epilogue          : TMEM -> registers -> per-warp smem transpose -> bias / act /
//                                   pos-enc / residual on 128-byte row segments -> coalesced stores
// TMEM map (512 columns): [0,256) two 128-column accumulators (the epilogue of tile i overlaps the
// mainloop of tile i+1); [256,512) four A stages of 32 hi + 32 lo columns.
// Rows of A may come from a strided / overlapping batched view (conv and STFT frames), addressed
// with a 3-D tensor map (k, row-in-batch, batch); M tiles never straddle a batch.
#include <cuda.h>

#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "kernels.cuh"

namespace vasr {

namespace {

constexpr int TBM = 128, TBN = 128, TBK = 32, STAGES = 4;
constexpr int TILE_BYTES = TBM * TBK * 4;            // 16 KB (A and W tiles are the same size)
constexpr int STAGE_BYTES = 3 * TILE_BYTES;          // A | W_hi | W_lo
constexpr int EPI_WARPS = 8;
constexpr int EPI_STAGE_BYTES = 32 * 128;            // one 32 x 32 fp32 chunk per epilogue warp
constexpr int BAR_OFFSET = STAGES * STAGE_BYTES + EPI_WARPS * EPI_STAGE_BYTES;
constexpr int SMEM_BYTES = BAR_OFFSET + 256 + 1024;  // + barriers + alignment slack
constexpr int TC_THREADS = 448;                      // 1 TMA + 1 MMA + 4 converter + 8 epilogue warps
constexpr uint32_t TMEM_COLS = 512;
constexpr uint32_t TMEM_A0 = 256;                    // first A column
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB of dynamic shared memory per CTA");

// barrier indices
constexpr int B_FULL = 0, B_CONV = STAGES, B_EMPTY = 2 * STAGES, B_TFULL = 3 * STAGES, B_TEMPTY = 3 * STAGES + 2;
constexpr int N_BARS = 3 * STAGES + 4;

// instruction descriptor (cute::UMMA::InstrDescriptor): c=F32 [4,6), a=TF32 [7,10), b=TF32 [10,13),
// K-major A and B, n_dim = N>>3 at [17,23), m_dim = M>>4 at [24,29)
__device__ __forceinline__ uint32_t make_idesc(uint32_t n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((n >> 3) << 17) | ((uint32_t)(TBM >> 4) << 24);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// bounded wait: a protocol bug traps (the launch fails with an error) instead of hanging the GPU.
// The clock is only started when the first probe fails: in steady state the barrier is already
// complete and the wait costs one try_wait (the MMA warp's per-stage bookkeeping is on the
// critical path of the tensor pipe, see DESIGN.md).
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity) {
  const long long t0 = clock64();
  while (!mbar_try(bar, parity))
    if (clock64() - t0 > 4000000000LL) __trap();
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (!mbar_try(bar, parity)) mbar_wait_slow(bar, parity);
}

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2,
                                            uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// L2 prefetch of a tile of the 3-D map: the persistent CTA knows its next tile a whole tile ahead, and an A tile
// that still sits in HBM costs a TMA load 2-3 k clocks — more than four 900-clock stages can hide
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* map, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global [%0, {%1, %2, %3}];" ::"l"(map), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}

// K-major, 128-byte swizzle, 8-row atoms 1024 B apart (cute::UMMA::SmemDescriptor, version 1)
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// D[tmem] (+)= A[tmem] · B[smem]ᵀ : 128 x N x 8, TF32 inputs, fp32 accumulate
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// true in exactly one lane of a converged warp.  The MMA operands are computed OUTSIDE the elected branch,
// from warp-uniform values only, so they sit in uniform registers: with operands derived from a
// per-thread value (e.g. the TMEM base read back from shared memory) ptxas wraps every UTCHMMA in an
// ELECT / R2UR.BROADCAST / BRA.U.ANY loop, ~85 clocks of dependent latency per MMA (round-1 trace).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
        "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
        "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}

// round-to-nearest TF32 (ties away), low 13 bits cleared
__device__ __forceinline__ uint32_t rna_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}

template <int ACT>
__device__ __forceinline__ float apply_act_t(float v) {
  if (ACT == ACT_GELU) return gelu_poly(v);
  if (ACT == ACT_SOFTPLUS) return softplus_t20(v);
  if (ACT == ACT_SIGMOID) return sigmoid_f(v);
  return v;
}

struct TcArgs {
  int64_t M, N, K;
  int64_t rows_per_batch;     // rows of A per batch (== M for a plain matrix)
  int64_t n_batches;
  int m_tiles_per_batch;
  int n_tiles;
  float* C;
  int64_t ldc;
  const float* bias;
  const float* q_scale;
  const float* q_zp;
  int act_from;
  const float* resid;
  int64_t ldr;
  const float* pe_time;
  const float* pe_freq;
  int pe_half;
  int prefetch;       // producer prefetches the next tile's A k-blocks into L2
  int dbg;            // debug (VASR_TC_DBG, garbage output): 1 = epilogue skips its TMEM loads, 2 = skips staging, math and stores
  int rotate_n;       // rotate the n-tile index by the round number (see tile_coords)
  int wres;           // pair kernel instantiated with WRES: pairs per n-tile.  Each pair keeps ONE n-tile: its W k-blocks
                      // are loaded once into the W halves of the stage ring (k-block kb always meets stage kb % nkb
                      // because nkb divides the ring) and only A streams afterwards
  long long* trace;   // debug: CTA 0 records clock64 at pipeline events (role, slot); NULL in production
  // LayerNorm folded into the projection (EPI_LNA): the rows of A are the LayerNorm's INPUT, W carries gamma, the
  // bias carries W beta; the converter thread that owns a row accumulates its sum and sum of squares while it
  // converts the k-blocks — of the row shifted by the mean c of its first 32 channels, which is also what it feeds the
  // tensor core — and leaves (rstd, -(mean - c) * rstd) in ln_stats; the epilogue applies
  // rstd * acc - (mean - c) * rstd * ln_s[n] + bias[n]  (ln_s[n] = sum_k W'[n, k]).
  const float* ln_s;
  float2* ln_stats;   // (M) scratch, one entry per row of A
  float ln_eps;
  // EPI_AMAX: per-row (max, argmax) over the columns each epilogue warp sees instead of the output itself:
  // slot p = 2 * n_tile + half at amax_val / amax_idx[p * M + row]
  float* amax_val;
  int32_t* amax_idx;
};
// epilogue variants (template bit mask)
constexpr int EPI_LNA = 1, EPI_AMAX = 2, EPI_GATE = 4;
// tile -> (m tile, n tile).  A persistent CTA takes tiles blockIdx.x, + gridDim.x, ...; with an n-tile
// count that divides the grid every tile of a CTA would have the same n index, and the CTAs that own
// the narrow last n-tile would do half the work of the others.  The n index is therefore rotated by
// the round number, so each CTA sees every n-tile in turn.
__device__ __forceinline__ void tile_coords(const TcArgs& g, int64_t tile64, int64_t units, int64_t* mt, int* nt) {
  // 32-bit arithmetic: tile counts are checked to fit by the launcher, and a 64-bit division is a ~150-clock
  // software routine that sat on the producer's and the MMA warp's per-tile path
  const uint32_t tile = (uint32_t)tile64, n_tiles = (uint32_t)g.n_tiles;
  const uint32_t m = tile / n_tiles;
  const uint32_t per = (uint32_t)units / n_tiles > 0 ? (uint32_t)units / n_tiles : 1u;
  *mt = m;
  *nt = (int)((tile - m * n_tiles + (g.rotate_n ? m / per : 0u)) % n_tiles);
}
// the time stamps inside the MMA warp cost it 50-100 clocks each (CS2R + store), enough to change what they
// measure; they are compiled in only with -DVASR_TC_TRACE_MMA
#ifdef VASR_TC_TRACE_MMA
#define MMA_TRACE(x) x
#else
#define MMA_TRACE(x)
#endif
constexpr int TRACE_SLOTS = 128;
constexpr int TRACE_ROLES = 16;
// pair kernel, per CTA: globaltimer at kernel entry, after griddepcontrol.wait, first accumulator complete, first
// tile stored, last accumulator complete, exit (tools/gemm_timeline.py)
constexpr int TRACE_CTA = 8;
__device__ __forceinline__ void trace_cta(const TcArgs& g, int slot) {
  if (g.trace) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g.trace[TRACE_ROLES * TRACE_SLOTS + TRACE_CTA * blockIdx.x + slot] = (long long)t;
  }
}
__device__ __forceinline__ void trace_ev(const TcArgs& g, int role, int idx) {
  if (g.trace && blockIdx.x == 0 && idx < TRACE_SLOTS) g.trace[role * TRACE_SLOTS + idx] = clock64();
}

// Epilogue of one warp over its tiles (shared by the single-CTA and the CTA-pair kernels).  PAIR: tiles are 256
// rows shared by the two CTAs of a cluster (this CTA owns rows rank*128 ..), tile index strides over pairs, and
// the accumulator-empty barrier lives in the leader CTA (arrive through its shared::cluster address).
template <int ACT, bool PE, bool RESID, bool QUANT, bool PAIR, int EPI = 0>
__device__ __forceinline__ void epilogue_loop(const TcArgs& g, uint8_t* stg, int warp, int lane, uint32_t first_tile,
                                              uint32_t tile_stride, uint32_t total_tiles32, uint32_t units, uint32_t rank,
                                              uint32_t bar_tfull0, uint32_t bar_tempty0_local,
                                              const float2* sstats = nullptr) {
  constexpr uint32_t tmem_base = 0u;
  constexpr uint32_t TM = PAIR ? 2 * TBM : TBM;          // rows of one tile
  auto BARF = [&](uint32_t acc) { return bar_tfull0 + 8u * acc; };
  auto arrive_empty = [&](uint32_t acc) {
    if (PAIR) {
      __syncwarp();
      if (lane == 0) {
        uint32_t r;
        asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(bar_tempty0_local + 8u * acc), "r"(0u));
        asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(r) : "memory");
      }
    } else {
      mbar_arrive(bar_tempty0_local + 8u * acc);
    }
  };
  // A warp reads two 32-row x 32-column chunks of the accumulator (thread = row), hands the accumulator
  // back as soon as both are in registers, transposes each chunk through its private 4 KB of shared
  // memory (16-byte chunks XOR-swizzled by row: conflict-free both ways) and then owns 128-byte row
  // segments: lane l handles columns 4*(l&7).. of rows (l>>3) + 4*i, so bias / activation / pos-enc /
  // residual and the store are coalesced.  Everything that does not depend on the accumulator (tile
  // coordinates in 32-bit arithmetic, bias, the residual rows of the first chunk) is fetched BEFORE the
  // wait for the accumulator: a trace showed 5.2 k clocks of epilogue per tile against 5.4 k of MMA.
  const int q = warp & 3;                         // TMEM lane quadrant this warp may read
  const int chalf = (warp - 6) >> 2;              // which two of the four 32-column chunks
    const int cc = lane & 7, rsub = lane >> 3;
  const uint32_t n_tiles = (uint32_t)g.n_tiles, mtpb = (uint32_t)g.m_tiles_per_batch;
  const uint32_t per = units / n_tiles > 0 ? units / n_tiles : 1u;
  const uint32_t rpb = (uint32_t)g.rows_per_batch;
  uint32_t it = 0;
  for (uint32_t tile = first_tile; tile < total_tiles32; tile += tile_stride, ++it) {
    // last tile of this CTA: the next kernel may be launched (programmatic dependent launch, common.cuh).  Not
    // earlier: a persistent grid that let its successor's CTAs sit resident in griddepcontrol.wait for its whole
    // run time would pay for it (see scan_seq_kernel).
    if (tile + tile_stride >= total_tiles32) pdl_trigger();
    const uint32_t mt = tile / n_tiles;
    const uint32_t nt = (tile % n_tiles + (g.rotate_n ? mt / per : 0u)) % n_tiles;
    const uint32_t batch = mt / mtpb;
    const uint32_t mi0 = (mt % mtpb) * TM + rank * TBM + q * 32;     // first row (within the batch) of this warp
    const uint32_t ncol0 = nt * TBN;
    const uint32_t nrem = (uint32_t)g.N - ncol0;
    const int nchunks = nrem >= (uint32_t)TBN ? 4 : (int)((nrem + 31) >> 5);   // chunks that hold real columns
    const uint32_t acc = it & 1u;
    const int c_begin = 2 * chalf, c_end = (2 * chalf + 2 < nchunks) ? 2 * chalf + 2 : nchunks;
    // this lane's four columns in chunk c_begin (+32 for the second chunk), and its row pointers
    const uint32_t n0 = ncol0 + c_begin * 32 + 4 * cc;
    const int64_t mrow0 = (int64_t)batch * rpb + mi0;               // global row of the warp's first row
    float* crow = g.C + mrow0 * g.ldc + n0;
    const float* rrow = RESID ? g.resid + mrow0 * g.ldr + n0 : nullptr;
    if constexpr ((EPI & EPI_AMAX) != 0) {
      // Greedy decode never needs the logits: thread = row keeps its 64 columns in registers, applies bias (and
      // the folded LayerNorm) per column and leaves (max, first index of the max) of what it saw; the collapse
      // kernel takes the best of a row's partials in column order (ties -> lowest index, as torch.argmax).
      static_assert(!PE && !RESID && !QUANT && ACT == ACT_NONE, "argmax epilogue: plain projection only");
      const uint32_t r = mi0 + lane;
      const int64_t grow = (int64_t)batch * rpb + r;
      const int64_t slot = ((int64_t)nt * 2 + chalf) * g.M + grow;
      mbar_wait(BARF(acc), (it >> 1) & 1u);
      tc_fence_after();
      if (c_begin >= c_end) {
        tc_fence_before();
        arrive_empty(acc);
        if (r < rpb) { g.amax_val[slot] = -INFINITY; g.amax_idx[slot] = -1; }
        continue;
      }
      uint32_t v0[32], v1[32];
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * TBN + c_begin * 32;
      tmem_ld32_issue(taddr, v0);
      if (c_begin + 1 < c_end) tmem_ld32_issue(taddr + 32, v1);
      float rs = 1.f, ms = 0.f;
      if (EPI & EPI_LNA) {       // left by this tile's converters in shared memory (the staging area is unused here)
        const float2 t = sstats[(it & 1u) * TBM + q * 32 + lane];
        rs = t.x; ms = t.y;
      }
      tmem_ld_wait();
      tc_fence_before();
      arrive_empty(acc);
      float best = -INFINITY;
      int bi = -1;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        if (c_begin + j >= c_end) break;
        const uint32_t nb = ncol0 + (c_begin + j) * 32;
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) {
          const uint32_t n = nb + 4 * k4;
          if (n >= (uint32_t)g.N) break;                               // N % 4 == 0: the group is valid as a whole
          const float4 b = g.bias ? __ldg(reinterpret_cast<const float4*>(g.bias + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
          float4 t = b;
          if (EPI & EPI_LNA) {
            const float4 sc = __ldg(reinterpret_cast<const float4*>(g.ln_s + n));
            t.x = fmaf(ms, sc.x, b.x); t.y = fmaf(ms, sc.y, b.y); t.z = fmaf(ms, sc.z, b.z); t.w = fmaf(ms, sc.w, b.w);
          }
          const float a0 = __uint_as_float(j == 0 ? v0[4 * k4] : v1[4 * k4]);
          const float a1 = __uint_as_float(j == 0 ? v0[4 * k4 + 1] : v1[4 * k4 + 1]);
          const float a2 = __uint_as_float(j == 0 ? v0[4 * k4 + 2] : v1[4 * k4 + 2]);
          const float a3 = __uint_as_float(j == 0 ? v0[4 * k4 + 3] : v1[4 * k4 + 3]);
          const float x0 = (EPI & EPI_LNA) ? fmaf(rs, a0, t.x) : a0 + t.x;
          const float x1 = (EPI & EPI_LNA) ? fmaf(rs, a1, t.y) : a1 + t.y;
          const float x2 = (EPI & EPI_LNA) ? fmaf(rs, a2, t.z) : a2 + t.z;
          const float x3 = (EPI & EPI_LNA) ? fmaf(rs, a3, t.w) : a3 + t.w;
          if (x0 > best || bi < 0) { best = x0; bi = (int)n; }
          if (x1 > best) { best = x1; bi = (int)n + 1; }
          if (x2 > best) { best = x2; bi = (int)n + 2; }
          if (x3 > best) { best = x3; bi = (int)n + 3; }
        }
      }
      if (r < rpb) { g.amax_val[slot] = best; g.amax_idx[slot] = bi; }
      continue;
    }
    float4 b4[2], qs4[2], qz4[2], pf4[2];
    bool col_ok[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const uint32_t n = n0 + 32 * j;
      col_ok[j] = (c_begin + j < c_end) && n < (uint32_t)g.N;       // N % 4 == 0: the group is valid as a whole
      b4[j] = qs4[j] = qz4[j] = pf4[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (!(EPI & EPI_LNA) && col_ok[j] && g.bias) b4[j] = __ldg(reinterpret_cast<const float4*>(g.bias + n));
      if (QUANT && col_ok[j]) {
        qs4[j] = __ldg(reinterpret_cast<const float4*>(g.q_scale + n));
        qz4[j] = __ldg(reinterpret_cast<const float4*>(g.q_zp + n));
      }
      if (PE && col_ok[j] && n >= (uint32_t)g.pe_half)
        pf4[j] = __ldg(reinterpret_cast<const float4*>(g.pe_freq + (n - g.pe_half)));
    }
    float4 r4[8];
    auto load_resid = [&](int j) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t rr = 4 * i + rsub;
        r4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (RESID && col_ok[j] && mi0 + rr < rpb)
          r4[i] = __ldg(reinterpret_cast<const float4*>(rrow + (int64_t)rr * g.ldr + 32 * j));
      }
    };
    if (RESID) load_resid(0);
    if (threadIdx.x == 192) trace_ev(g, 5, (int)it);     // ready to take tile `it`
    mbar_wait(BARF(acc), (it >> 1) & 1u);
    if (threadIdx.x == 192) trace_ev(g, 6, (int)it);     // accumulator complete
    tc_fence_after();
    if (c_begin >= c_end) {       // nothing of this tile belongs to this warp: hand the accumulator back
      tc_fence_before();
      arrive_empty(acc);
      continue;
    }
    uint32_t v0[32], v1[32];
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * TBN + c_begin * 32;
    if (!(g.dbg & 1)) {
      tmem_ld32_issue(taddr, v0);
      if (c_begin + 1 < c_end) tmem_ld32_issue(taddr + 32, v1);
      float2 own = make_float2(1.f, 0.f);
      if constexpr ((EPI & EPI_LNA) != 0) {
        if (mi0 + lane < rpb) own = __ldcg(g.ln_stats + mrow0 + lane);   // left by this tile's converters
      }
      tmem_ld_wait();
      if constexpr ((EPI & EPI_LNA) != 0) {
        // thread = row:  rstd * acc + (-(mean - c) * rstd * s[n] + bias[n])  on the chunks as they sit in registers
        const u64 rs2 = pack2(own.x, own.x), ms2 = pack2(own.y, own.y);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (c_begin + j >= c_end) break;
          const uint32_t nb = ncol0 + (c_begin + j) * 32;
#pragma unroll
          for (int k4 = 0; k4 < 8; ++k4) {
            if (nb + 4 * k4 >= (uint32_t)g.N) break;
            const float4 sc = __ldg(reinterpret_cast<const float4*>(g.ln_s + nb + 4 * k4));
            const float4 bc = g.bias ? __ldg(reinterpret_cast<const float4*>(g.bias + nb + 4 * k4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            uint32_t* v = j == 0 ? v0 : v1;
            u64 a = pack2(__uint_as_float(v[4 * k4]), __uint_as_float(v[4 * k4 + 1]));
            u64 b = pack2(__uint_as_float(v[4 * k4 + 2]), __uint_as_float(v[4 * k4 + 3]));
            a = fma2(rs2, a, fma2(ms2, pack2(sc.x, sc.y), pack2(bc.x, bc.y)));
            b = fma2(rs2, b, fma2(ms2, pack2(sc.z, sc.w), pack2(bc.z, bc.w)));
            float f0, f1, f2, f3;
            unpack2(a, f0, f1); unpack2(b, f2, f3);
            v[4 * k4] = __float_as_uint(f0); v[4 * k4 + 1] = __float_as_uint(f1);
            v[4 * k4 + 2] = __float_as_uint(f2); v[4 * k4 + 3] = __float_as_uint(f3);
          }
        }
      }
    } else {
#pragma unroll
      for (int k = 0; k < 32; ++k) v0[k] = v1[k] = 0u;
    }
    tc_fence_before();
    arrive_empty(acc);                  // this warp's share of the accumulator is in registers
    if (threadIdx.x == 192) trace_ev(g, 7, (int)it);
    if (g.dbg & 2) continue;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      if (c_begin + j >= c_end) break;
      {
        uint8_t* srow = stg + lane * 128;
#pragma unroll
        for (int k = 0; k < 8; ++k)
          *reinterpret_cast<uint4*>(srow + ((k ^ (lane & 7)) << 4)) =
              j == 0 ? make_uint4(v0[4 * k], v0[4 * k + 1], v0[4 * k + 2], v0[4 * k + 3])
                     : make_uint4(v1[4 * k], v1[4 * k + 1], v1[4 * k + 2], v1[4 * k + 3]);
      }
      __syncwarp();
      if (threadIdx.x == 192 && j == 0) trace_ev(g, 8, (int)it);
      const uint32_t n = n0 + 32 * j;
      const bool act_on = ACT != ACT_NONE && n >= (uint32_t)g.act_from;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t rr = 4 * i + rsub;
        float4 x = *reinterpret_cast<const float4*>(stg + rr * 128 + ((cc ^ (rr & 7)) << 4));
        if constexpr ((EPI & EPI_LNA) == 0) { x.x += b4[j].x; x.y += b4[j].y; x.z += b4[j].z; x.w += b4[j].w; }
        if (QUANT) {
          x.x = fake_quant_u8(x.x, qs4[j].x, qz4[j].x); x.y = fake_quant_u8(x.y, qs4[j].y, qz4[j].y);
          x.z = fake_quant_u8(x.z, qs4[j].z, qz4[j].z); x.w = fake_quant_u8(x.w, qs4[j].w, qz4[j].w);
        }
        if (act_on) {
          if (ACT == ACT_GELU) {
            gelu_poly2(x.x, x.y);
            gelu_poly2(x.z, x.w);
          } else {
            x.x = apply_act_t<ACT>(x.x); x.y = apply_act_t<ACT>(x.y);
            x.z = apply_act_t<ACT>(x.z); x.w = apply_act_t<ACT>(x.w);
          }
        }
        if (PE) {
          float4 p4 = pf4[j];
          if (n < (uint32_t)g.pe_half && col_ok[j] && mi0 + rr < rpb)
            p4 = __ldg(reinterpret_cast<const float4*>(g.pe_time + (int64_t)(mi0 + rr) * g.pe_half + n));
          x.x += p4.x; x.y += p4.y; x.z += p4.z; x.w += p4.w;
        }
        if (RESID) { x.x += r4[i].x; x.y += r4[i].y; x.z += r4[i].z; x.w += r4[i].w; }
        if (col_ok[j] && mi0 + rr < rpb) *reinterpret_cast<float4*>(crow + (int64_t)rr * g.ldc + 32 * j) = x;
      }
      __syncwarp();               // the staging chunk is rewritten by the next chunk
      if (RESID && j == 0 && c_begin + 1 < c_end) load_resid(1);
      if (threadIdx.x == 192 && j == 0) trace_ev(g, 9, (int)it);
    }
  }
}

// Epilogue of the 192-column pair kernel (plain projections, optional residual): six 32-column chunks per tile,
// three per warp.  Two chunks are read at once as above; the first is transposed and stored, then its registers
// take the third chunk and only then is the accumulator handed back (the tile's MMAs take 13.8 k clocks, the
// epilogue has time).  Same staging, same coalesced 128-byte row segments as epilogue_loop.
template <int ACT, bool RESID, int EPI = 0>
__device__ __forceinline__ void epilogue_loop192(const TcArgs& g, uint8_t* stg, float2* rowfac, const float2* sstats, int warp, int lane, uint32_t first_tile,
                                                 uint32_t tile_stride, uint32_t total_tiles32, uint32_t rank,
                                                 uint32_t bar_tfull0, uint32_t bar_tempty0_local) {
  constexpr uint32_t tmem_base = 0u;
  constexpr uint32_t TN = 192, TM = 2 * TBM;
  auto arrive_empty = [&](uint32_t acc) {
    __syncwarp();
    if (lane == 0) {
      uint32_t r;
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(bar_tempty0_local + 8u * acc), "r"(0u));
      asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(r) : "memory");
    }
  };
  const int q = warp & 3;
  const int chalf = (warp - 6) >> 2;              // which three of the six 32-column chunks
  const int cc = lane & 7, rsub = lane >> 3;
  const uint32_t n_tiles = (uint32_t)g.n_tiles, mtpb = (uint32_t)g.m_tiles_per_batch;
  const uint32_t rpb = (uint32_t)g.rows_per_batch;
  uint32_t it = 0;
  for (uint32_t tile = first_tile; tile < total_tiles32; tile += tile_stride, ++it) {
    if (tile + tile_stride >= total_tiles32) pdl_trigger();        // last tile of this CTA (see epilogue_loop)
    const uint32_t mt = tile / n_tiles, nt = tile - mt * n_tiles;
    const uint32_t batch = mt / mtpb;
    const uint32_t mi0 = (mt % mtpb) * TM + rank * TBM + q * 32;
    const uint32_t ncol0 = nt * TN;
    const uint32_t nrem = (uint32_t)g.N - ncol0;
    const int nchunks = nrem >= TN ? 6 : (int)((nrem + 31) >> 5);
    const uint32_t acc = it & 1u;
    const int c_begin = 3 * chalf, c_end = (c_begin + 3 < nchunks) ? c_begin + 3 : nchunks;
    const uint32_t n0 = ncol0 + c_begin * 32 + 4 * cc;
    const int64_t mrow0 = (int64_t)batch * rpb + mi0;
    float* crow = g.C + mrow0 * g.ldc + n0;
    const float* rrow = RESID ? g.resid + mrow0 * g.ldr + n0 : nullptr;
    float4 b4[3];
    bool col_ok[3];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const uint32_t n = n0 + 32 * j;
      col_ok[j] = (c_begin + j < c_end) && n < (uint32_t)g.N;
      b4[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (col_ok[j] && g.bias) b4[j] = __ldg(reinterpret_cast<const float4*>(g.bias + n));
    }
    if constexpr ((EPI & EPI_GATE) != 0) {
      // GatedFusion (attention.py:191-220): the weight rows were permuted at pack time so that the three chunks of
      // this warp are gate logits | local_proj | global_proj of the SAME 32 channels (64 * nt + 32 * chalf ..); the
      // mix s * l + (1 - s) * t happens here and only the 192 mixed channels are written (C is M x N/3).
      static_assert(!RESID && ACT == ACT_NONE && !(EPI & EPI_LNA), "gate epilogue: plain stacked projection");
      float* orow = g.C + mrow0 * g.ldc + nt * 64 + chalf * 32 + 4 * cc;
      mbar_wait(bar_tfull0 + 8u * acc, (it >> 1) & 1u);
      tc_fence_after();
      uint32_t v0[32], v1[32];
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * TN + c_begin * 32;
      tmem_ld32_issue(taddr, v0);
      tmem_ld32_issue(taddr + 32, v1);
      tmem_ld_wait();
      float4 gx[8], lx[8];
      auto take = [&](const uint32_t (&v)[32], int j, float4 (&o)[8]) {
        uint8_t* srow = stg + lane * 128;
#pragma unroll
        for (int k = 0; k < 8; ++k)
          *reinterpret_cast<uint4*>(srow + ((k ^ (lane & 7)) << 4)) = make_uint4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint32_t rr = 4 * i + rsub;
          float4 x = *reinterpret_cast<const float4*>(stg + rr * 128 + ((cc ^ (rr & 7)) << 4));
          x.x += b4[j].x; x.y += b4[j].y; x.z += b4[j].z; x.w += b4[j].w;
          o[i] = x;
        }
        __syncwarp();
      };
      take(v0, 0, gx);
      tmem_ld32_issue(taddr + 64, v0);
      tmem_ld_wait();
      tc_fence_before();
      arrive_empty(acc);
      take(v1, 1, lx);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        gx[i].x = sigmoid_f(gx[i].x); gx[i].y = sigmoid_f(gx[i].y); gx[i].z = sigmoid_f(gx[i].z); gx[i].w = sigmoid_f(gx[i].w);
      }
      {
        uint8_t* srow = stg + lane * 128;
#pragma unroll
        for (int k = 0; k < 8; ++k)
          *reinterpret_cast<uint4*>(srow + ((k ^ (lane & 7)) << 4)) = make_uint4(v0[4 * k], v0[4 * k + 1], v0[4 * k + 2], v0[4 * k + 3]);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint32_t rr = 4 * i + rsub;
          float4 t = *reinterpret_cast<const float4*>(stg + rr * 128 + ((cc ^ (rr & 7)) << 4));
          t.x += b4[2].x; t.y += b4[2].y; t.z += b4[2].z; t.w += b4[2].w;
          float4 o;
          o.x = gx[i].x * lx[i].x + (1.0f - gx[i].x) * t.x;
          o.y = gx[i].y * lx[i].y + (1.0f - gx[i].y) * t.y;
          o.z = gx[i].z * lx[i].z + (1.0f - gx[i].z) * t.z;
          o.w = gx[i].w * lx[i].w + (1.0f - gx[i].w) * t.w;
          if (mi0 + rr < rpb) *reinterpret_cast<float4*>(orow + (int64_t)rr * g.ldc) = o;
        }
        __syncwarp();
      }
      continue;
    }
    float4 r4[8];
    auto load_resid = [&](int j) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t rr = 4 * i + rsub;
        r4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (RESID && col_ok[j] && mi0 + rr < rpb)
          r4[i] = __ldg(reinterpret_cast<const float4*>(rrow + (int64_t)rr * g.ldr + 32 * j));
      }
    };
    if (RESID) {
      load_resid(0);
      // the residual rows of the other two chunks are fetched after the accumulator has been handed back, with
      // nothing left to hide a trip to HBM behind (tools/gemm_timeline.py: 6 us from "accumulator complete" to
      // "tile stored", all of it exposed at the end of a launch): start them on their way to L2 now
      if (cc == 0) {
#pragma unroll
        for (int j = 1; j < 3; ++j)
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint32_t rr = 4 * i + rsub;
            if (col_ok[j] && mi0 + rr < rpb)
              asm volatile("prefetch.global.L2 [%0];" ::"l"(rrow + (int64_t)rr * g.ldr + 32 * j));
          }
      }
    }
    mbar_wait(bar_tfull0 + 8u * acc, (it >> 1) & 1u);
    if (warp == 6 && lane == 0) { if (it == 0) trace_cta(g, 2); trace_cta(g, 4); }
    tc_fence_after();
    if (c_begin >= c_end) {
      tc_fence_before();
      arrive_empty(acc);
      continue;
    }
    uint32_t v0[32], v1[32];
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * TN + c_begin * 32;
    tmem_ld32_issue(taddr, v0);
    if (c_begin + 1 < c_end) tmem_ld32_issue(taddr + 32, v1);
    // EPI_LNA: the thread that owns a row of the accumulator fetches the row's (rstd, -(mean - c) * rstd) and leaves
    // them in this warp's row-factor table; after the transpose a lane picks up the factors of each of its rows
    // next to the row segment itself (no long-lived registers, no per-column loads: the GELU epilogue is the
    // critical path of ffn.0, every instruction here is paid in full)
    float4 s4[3];
    if constexpr ((EPI & EPI_LNA) != 0) {
      // the converters' table is double-buffered by tile parity; it is copied before the accumulator is handed
      // back, so the converters of tile it + 2 (which need that hand-over) cannot overwrite what is still in use
      rowfac[lane] = sstats[(it & 1u) * TBM + q * 32 + lane];          // ordered by the __syncwarp of the first transpose
#pragma unroll
      for (int j = 0; j < 3; ++j)
        s4[j] = col_ok[j] ? __ldg(reinterpret_cast<const float4*>(g.ln_s + n0 + 32 * j)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    tmem_ld_wait();
    // chunk j of this warp: registers -> swizzled staging -> 128-byte row segments (+ bias, residual) -> global
    auto emit = [&](const uint32_t (&v)[32], int j) {
      uint8_t* srow = stg + lane * 128;
#pragma unroll
      for (int k = 0; k < 8; ++k)
        *reinterpret_cast<uint4*>(srow + ((k ^ (lane & 7)) << 4)) = make_uint4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint32_t rr = 4 * i + rsub;
        float4 x = *reinterpret_cast<const float4*>(stg + rr * 128 + ((cc ^ (rr & 7)) << 4));
        if constexpr ((EPI & EPI_LNA) != 0) {
          // packed: a 3-register scalar FFMA occupies the FMA pipe as long as an FFMA2 does, and that pipe is what
          // the GELU epilogue is bound by
          const float2 f = rowfac[rr];
          const u64 rs2 = pack2(f.x, f.x), ms2 = pack2(f.y, f.y);
          const u64 lo = fma2(rs2, pack2(x.x, x.y), fma2(ms2, pack2(s4[j].x, s4[j].y), pack2(b4[j].x, b4[j].y)));
          const u64 hi = fma2(rs2, pack2(x.z, x.w), fma2(ms2, pack2(s4[j].z, s4[j].w), pack2(b4[j].z, b4[j].w)));
          unpack2(lo, x.x, x.y);
          unpack2(hi, x.z, x.w);
        } else {
          const u64 lo = add2(pack2(x.x, x.y), pack2(b4[j].x, b4[j].y)), hi = add2(pack2(x.z, x.w), pack2(b4[j].z, b4[j].w));
          unpack2(lo, x.x, x.y);
          unpack2(hi, x.z, x.w);
        }
        if (ACT != ACT_NONE && n0 + 32 * j >= (uint32_t)g.act_from) {
          if (ACT == ACT_GELU) {
            gelu_poly2(x.x, x.y);
            gelu_poly2(x.z, x.w);
          } else {
            x.x = apply_act_t<ACT>(x.x); x.y = apply_act_t<ACT>(x.y);
            x.z = apply_act_t<ACT>(x.z); x.w = apply_act_t<ACT>(x.w);
          }
        }
        if (RESID) { x.x += r4[i].x; x.y += r4[i].y; x.z += r4[i].z; x.w += r4[i].w; }
        if (col_ok[j] && mi0 + rr < rpb) *reinterpret_cast<float4*>(crow + (int64_t)rr * g.ldc + 32 * j) = x;
      }
      __syncwarp();
    };
    emit(v0, 0);
    const bool has2 = c_begin + 2 < c_end;
    if (has2) {
      tmem_ld32_issue(taddr + 64, v0);
      tmem_ld_wait();
    }
    tc_fence_before();
    arrive_empty(acc);                  // everything this warp needs of the accumulator is in registers
    if (c_begin + 1 < c_end) {
      if (RESID) load_resid(1);
      emit(v1, 1);
    }
    if (has2) {
      if (RESID) load_resid(2);
      emit(v0, 2);
    }
    if (warp == 6 && lane == 0 && it == 0) trace_cta(g, 3);
  }
}

template <int ACT, bool PE, bool RESID, bool QUANT>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmWh,
               const __grid_constant__ CUtensorMap tmWl, const TcArgs g) {
  extern __shared__ uint8_t smem_raw[];
  // keep the pointer derived from smem_raw (no integer round trip) so accesses compile to LDS/STS
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BAR_OFFSET);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + N_BARS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const uint32_t stage0 = smem_u32(smem);

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(BAR(B_FULL + s), 1);       // producer's expect_tx arrive
      mbar_init(BAR(B_CONV + s), 128);     // every converter thread
      mbar_init(BAR(B_EMPTY + s), 1);      // tcgen05.commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(BAR(B_TFULL + a), 1);               // tcgen05.commit
      mbar_init(BAR(B_TEMPTY + a), EPI_WARPS * 32); // every epilogue thread
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // the whole TMEM (512 columns) is allocated, so the base can only be 0: using the literal keeps every
  // TMEM address warp-uniform for the compiler (see elect_one)
  if (*tmem_slot != 0u) __trap();
  constexpr uint32_t tmem_base = 0u;
  pdl_wait();          // prologue done; global memory from here on (programmatic dependent launch, common.cuh)

  const int nkb = (int)((g.K + TBK - 1) / TBK);
  const int64_t total_tiles = (int64_t)g.n_tiles * g.m_tiles_per_batch * g.n_batches;
  const int64_t UNITS = gridDim.x;
  if (threadIdx.x == 0) trace_cta(g, 0);

  if (warp == 0) {
    // ===================== TMA producer =====================
    // (whole warp runs the loop so that coordinates and addresses stay warp-uniform; one lane issues)
    uint32_t stage = 0, phase = 0;
    int tr_i = 0;
    for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      int nt;
      int64_t mt;
      tile_coords(g, tile, UNITS, &mt, &nt);
      const int batch = (int)((uint32_t)mt / (uint32_t)g.m_tiles_per_batch);
      const int mi0 = (int)((uint32_t)mt % (uint32_t)g.m_tiles_per_batch) * TBM;
      if (g.prefetch && tile + gridDim.x < total_tiles) {
        int nnt;
        int64_t nmt;
        tile_coords(g, tile + gridDim.x, UNITS, &nmt, &nnt);
        const int nbatch = (int)((uint32_t)nmt / (uint32_t)g.m_tiles_per_batch);
        const int nmi0 = (int)((uint32_t)nmt % (uint32_t)g.m_tiles_per_batch) * TBM;
        if (elect_one())
          for (int kb = 0; kb < nkb; ++kb) tma_prefetch_3d(&tmA, kb * TBK, nmi0, nbatch);
        __syncwarp();
      }
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(BAR(B_EMPTY + stage), phase ^ 1);
        if (lane == 0) trace_ev(g, 0, tr_i);
        ++tr_i;
        const uint32_t sb = stage0 + stage * STAGE_BYTES;
        if (elect_one()) {
          mbar_expect_tx(BAR(B_FULL + stage), 3 * TILE_BYTES);
          tma_load_3d(sb, &tmA, kb * TBK, mi0, batch, BAR(B_FULL + stage));
          tma_load_2d(sb + TILE_BYTES, &tmWh, kb * TBK, nt * TBN, BAR(B_FULL + stage));
          tma_load_2d(sb + 2 * TILE_BYTES, &tmWl, kb * TBK, nt * TBN, BAR(B_FULL + stage));
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    uint32_t stage = 0, phase = 0;
    int64_t it = 0;
    int tr_i = 0;
    for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      int nt;
      int64_t mt_unused;
      tile_coords(g, tile, UNITS, &mt_unused, &nt);
      // columns of this tile that exist, rounded up to the MMA's N granularity (16)
      int64_t nrem = g.N - (int64_t)nt * TBN;
      const uint32_t n_mma = nrem >= TBN ? (uint32_t)TBN : (uint32_t)((nrem + 15) & ~15LL);
      const uint32_t idesc = make_idesc(n_mma);
      const uint32_t acc = (uint32_t)(it & 1);
      mbar_wait(BAR(B_TEMPTY + acc), (uint32_t)((it >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * TBN;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(BAR(B_FULL + stage), phase);    // W tiles landed (async proxy)
        mbar_wait(BAR(B_CONV + stage), phase);    // A hi/lo are in TMEM
        tc_fence_after();
        if (lane == 0) trace_ev(g, 3, tr_i);
        const uint32_t sb = stage0 + stage * STAGE_BYTES;
        const uint64_t db_hi = umma_desc(sb + TILE_BYTES), db_lo = umma_desc(sb + 2 * TILE_BYTES);
        const uint32_t a_hi = tmem_base + TMEM_A0 + stage * 64, a_lo = a_hi + 32;
        if (elect_one()) {
#pragma unroll
          for (int k4 = 0; k4 < TBK / 8; ++k4) {
            const uint64_t adv = (uint64_t)(k4 * 2);   // 8 tf32 = 32 bytes = 2 x 16-byte units
            umma_tf32_ts(tmem_d, a_lo + 8 * k4, db_hi + adv, idesc, (kb | k4) != 0);
            umma_tf32_ts(tmem_d, a_hi + 8 * k4, db_lo + adv, idesc, 1);
            umma_tf32_ts(tmem_d, a_hi + 8 * k4, db_hi + adv, idesc, 1);
          }
          umma_commit(BAR(B_EMPTY + stage));
          if (kb == nkb - 1) umma_commit(BAR(B_TFULL + acc));
          trace_ev(g, 4, tr_i);
        }
        ++tr_i;
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp < 6) {
    // ===================== converters: A row -> (hi, lo) -> TMEM =====================
    // Thread = one row of the tile = one TMEM lane (a warp may touch lanes 32*(warp%4) .. +31).
    // Row r of the swizzled tile is 128 contiguous bytes whose 16-byte chunk c sits at c ^ (r & 7):
    // the eight lanes of a load phase hit eight different chunks, so the reads are conflict-free.
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + TMEM_A0;
    uint32_t stage = 0, phase = 0;
    int tr_i = 0;
    for (int64_t tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(BAR(B_FULL + stage), phase);
        if (threadIdx.x == 64) trace_ev(g, 1, tr_i);
        const uint8_t* arow = smem + stage * STAGE_BYTES + row * 128;
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 v = *reinterpret_cast<const float4*>(arow + ((c ^ (row & 7)) << 4));
          hi[4 * c + 0] = rna_tf32(v.x); lo[4 * c + 0] = rna_tf32(v.x - __uint_as_float(hi[4 * c + 0]));
          hi[4 * c + 1] = rna_tf32(v.y); lo[4 * c + 1] = rna_tf32(v.y - __uint_as_float(hi[4 * c + 1]));
          hi[4 * c + 2] = rna_tf32(v.z); lo[4 * c + 2] = rna_tf32(v.z - __uint_as_float(hi[4 * c + 2]));
          hi[4 * c + 3] = rna_tf32(v.w); lo[4 * c + 3] = rna_tf32(v.w - __uint_as_float(hi[4 * c + 3]));
        }
        // the TMEM slot of this stage was last read by MMAs whose commit released `empty[stage]`,
        // which the producer waited on before the TMA that completed `full[stage]`
        tc_fence_after();
        tmem_st32(lane_addr + stage * 64, hi);
        tmem_st32(lane_addr + stage * 64 + 32, lo);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        mbar_arrive(BAR(B_CONV + stage));
        if (threadIdx.x == 64) trace_ev(g, 2, tr_i);
        ++tr_i;
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue =====================
    epilogue_loop<ACT, PE, RESID, QUANT, false>(g, smem + STAGES * STAGE_BYTES + (warp - 6) * EPI_STAGE_BYTES, warp, lane,
                                                blockIdx.x, gridDim.x, (uint32_t)total_tiles, (uint32_t)UNITS, 0u,
                                                BAR(B_TFULL), BAR(B_TEMPTY));
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) trace_cta(g, 7);
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
  }
}

// =============================================================================================
// CTA-pair version (cta_group::2).  ncu on the single-CTA kernel above: the tensor pipe is 48 % busy
// and shared memory 77 % — per 32-deep k-step a CTA moves 896 wavefronts (TMA writes of A and of
// both W tiles, the converter's read of A, three MMA reads of W) against 768 clocks of MMA.  Two CTAs
// of a cluster (one TPC) therefore share a 256 x 128 tile: each holds its own 128 rows of A (in its
// own TMEM) and HALF of the W tile; one tcgen05.mma.cta_group::2 issued by the leader drives both
// tensor cores, and each SM's shared memory sees 576 wavefronts per k-step (A in + A read + half of W
// in + half of the W reads).  Barriers: the W-full, conversion-done and accumulator-empty barriers
// live in the leader and are signalled remotely by the peer; stage-empty and accumulator-full are
// multicast to both CTAs by tcgen05.commit.
// =============================================================================================
constexpr int P_STAGE_BYTES = 2 * TILE_BYTES;                         // A (16 KB) | W_hi half (8 KB) | W_lo half (8 KB)
constexpr int P_STAGES = 6;                                          // shared-memory stages (32 KB each)
constexpr int P_ASLOTS = 4;                                          // A (hi | lo) slots in TMEM, 64 columns each
constexpr int P_BAR_OFFSET = P_STAGES * P_STAGE_BYTES + EPI_WARPS * EPI_STAGE_BYTES;
constexpr int P_SMEM_BYTES = P_BAR_OFFSET + 512 + 1024;
static_assert(P_SMEM_BYTES <= 232448, "exceeds the 227 KB of dynamic shared memory per CTA");
// barrier indices (per CTA; the leader's copies of WFULL / CONV / TEMPTY are the ones in use)
constexpr int PB_AFULL = 0, PB_WFULL = P_STAGES, PB_CONV = 2 * P_STAGES, PB_EMPTY = 3 * P_STAGES,
              PB_TFULL = 4 * P_STAGES, PB_TEMPTY = 4 * P_STAGES + 2, PB_AFREE = 4 * P_STAGES + 4;
constexpr int P_NBARS = 4 * P_STAGES + 4 + P_ASLOTS;

// The same kernel with 192-column tiles (TN = 192), for N = 192 / 576: with 128-column tiles those projections end
// in a 64-column tile whose k-blocks complete at the pace of the control path (converter and MMA warps, ~770
// clocks) although their MMAs take 384 — half the tile time at half the tensor rate, and A loaded and converted
// twice per row block.  One 192-column MMA per k-step (96 clocks) is tensor-bound again.  Costs: 2 x 192
// accumulator columns leave room for two A slots only, and a stage grows to 40 KB (four of them).
template <int TN>
struct PairCfg {
  static constexpr int W_HALF_BYTES = (TN / 2) * TBK * 4;              // one CTA's rows of W_hi (or W_lo) of a stage
  static constexpr int STAGE_BYTES = TILE_BYTES + 2 * W_HALF_BYTES;     // A | W_hi half | W_lo half
  static constexpr int STAGES = TN == 128 ? 6 : 4;
  static constexpr int ASLOTS = TN == 128 ? 4 : 2;
  static constexpr uint32_t A0 = 2 * TN;                               // first A column (two accumulators before it)
  static constexpr int BAR_OFFSET = STAGES * STAGE_BYTES + EPI_WARPS * EPI_STAGE_BYTES;
  static constexpr int ROWFAC_OFFSET = BAR_OFFSET + 512;                // TN = 192: 32 x float2 per epilogue warp (EPI_LNA)
  static constexpr int SMEM_BYTES = BAR_OFFSET + 512 + (TN == 192 ? EPI_WARPS * 256 + 2 * TBM * 8 : 0) + 1024;
  static constexpr int AFULL = 0, WFULL = STAGES, CONV = 2 * STAGES, EMPTY = 3 * STAGES, TFULL = 4 * STAGES,
                       TEMPTY = 4 * STAGES + 2, AFREE = 4 * STAGES + 4, NBARS = 4 * STAGES + 4 + ASLOTS;
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB of dynamic shared memory per CTA");
  static_assert(A0 + ASLOTS * 64 <= 512, "tensor memory");
};
static_assert(PairCfg<128>::STAGE_BYTES == P_STAGE_BYTES && PairCfg<128>::SMEM_BYTES == P_SMEM_BYTES, "TN = 128 is the layout above");

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ bool mbar_try_cluster(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __noinline__ void mbar_wait_cluster_slow(uint32_t bar, uint32_t parity) {
  const long long t0 = clock64();
  while (!mbar_try_cluster(bar, parity))
    if (clock64() - t0 > 4000000000LL) __trap();
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  if (!mbar_try_cluster(bar, parity)) mbar_wait_cluster_slow(bar, parity);
}
// TMA load whose completion bytes are credited to a barrier of the LEADER CTA of the pair
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, int c0, int c1,
                                                 uint32_t leader_bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_ts_pair(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"((uint16_t)3)
      : "memory");
}

template <int ACT, bool PE, bool RESID, bool QUANT, bool WRES = false, int TN = 128, int EPI = 0>
#ifdef VASR_TC_MAXNREG
__global__ void __cluster_dims__(2, 1, 1) __maxnreg__(144)
#else
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
#endif
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmWh,
                const __grid_constant__ CUtensorMap tmWl, const TcArgs g) {
  // the tile-width dependent layout, under the names the body uses (they shadow the TN = 128 globals)
  using Cfg = PairCfg<TN>;
  constexpr int TBN = TN;
  constexpr int P_STAGE_BYTES = Cfg::STAGE_BYTES, P_STAGES = Cfg::STAGES, P_ASLOTS = Cfg::ASLOTS;
  constexpr int P_BAR_OFFSET = Cfg::BAR_OFFSET, P_NBARS = Cfg::NBARS;
  constexpr int PB_AFULL = Cfg::AFULL, PB_WFULL = Cfg::WFULL, PB_CONV = Cfg::CONV, PB_EMPTY = Cfg::EMPTY,
                PB_TFULL = Cfg::TFULL, PB_TEMPTY = Cfg::TEMPTY, PB_AFREE = Cfg::AFREE;
  constexpr uint32_t TMEM_A0 = Cfg::A0;
  constexpr int W_HALF_BYTES = Cfg::W_HALF_BYTES;
  static_assert(!(WRES && TN != 128), "the W-resident schedule exists for 128-column tiles only");
  // EPI_LNA: where the converters leave a tile's row statistics for its epilogue.  Shared memory (2 x 128 float2,
  // by tile parity) where there is room — the 192-column layout, and the argmax epilogue, whose transpose staging
  // is unused; global scratch otherwise (the epilogue then pays an L2 round trip per tile after the accumulator
  // arrives: ~7 us on ffn.0 when it still took that route).
  constexpr bool SSTATS = (EPI & EPI_LNA) != 0 && (TN == 192 || (EPI & EPI_AMAX) != 0);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + P_BAR_OFFSET);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + P_NBARS);

  if (threadIdx.x == 0) {   // descriptor fetches off the first TMA's critical path (kernel parameters: no dependency)
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmWh)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmWl)) : "memory");
  }
  if (threadIdx.x == 0) trace_cta(g, 0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  const uint32_t stage0 = smem_u32(smem);
  float2* sstats = reinterpret_cast<float2*>(TN == 192 ? smem + Cfg::ROWFAC_OFFSET + EPI_WARPS * 256
                                                       : smem + P_STAGES * P_STAGE_BYTES);

  if (threadIdx.x == 0) {
    for (int s = 0; s < P_STAGES; ++s) {
      mbar_init(BAR(PB_AFULL + s), 1);       // local: this CTA's A tile
      mbar_init(BAR(PB_WFULL + s), 1);       // leader: both W halves (one expect_tx arrive by the leader)
      mbar_init(BAR(PB_CONV + s), 8);        // leader: one arrive per converter warp of both CTAs
      mbar_init(BAR(PB_EMPTY + s), 1);       // local, multicast tcgen05.commit
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(BAR(PB_TFULL + a), 1);                    // local, multicast tcgen05.commit
      mbar_init(BAR(PB_TEMPTY + a), 2 * EPI_WARPS);       // leader: one arrive per epilogue warp of both CTAs
    }
    for (int a = 0; a < P_ASLOTS; ++a) mbar_init(BAR(PB_AFREE + a), 1);   // local, multicast tcgen05.commit
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();           // both CTAs' barriers are initialised before anyone signals across
  tc_fence_after();
  // the whole TMEM (512 columns) is allocated, so the base can only be 0: using the literal keeps every
  // TMEM address warp-uniform for the compiler (see elect_one)
  if (*tmem_slot != 0u) __trap();
  constexpr uint32_t tmem_base = 0u;
  // barriers, tensor memory and the cluster handshake are set up; from here on global memory is touched, which
  // has to wait for the previous kernel (programmatic dependent launch, common.cuh)
  if (threadIdx.x == 0) trace_cta(g, 6);
  pdl_wait();
  if (threadIdx.x == 0) trace_cta(g, 1);

  const int nkb = (int)((g.K + TBK - 1) / TBK);
  const int64_t total_tiles = (int64_t)g.n_tiles * g.m_tiles_per_batch * g.n_batches;   // pair tiles (256 rows)
  const int64_t pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int64_t UNITS = npairs;
  // tile walk of this pair: round-robin over all tiles, or (W resident) a fixed n-tile and every wres-th m-tile
  int64_t first_tile = pair, tile_stride = npairs;
  if (WRES) {
    const int64_t slot = pair / g.n_tiles, nt_own = pair % g.n_tiles;
    first_tile = slot < g.wres ? slot * g.n_tiles + nt_own : total_tiles;
    tile_stride = (int64_t)g.wres * g.n_tiles;
  }

  if (warp == 0) {
    // ===================== TMA producer (both CTAs) =====================
    uint32_t stage = 0, phase = 0, cnt = 0;
    int tr_i = 0;
    for (int64_t tile = first_tile; tile < total_tiles; tile += tile_stride) {
      int nt;
      int64_t mt;
      tile_coords(g, tile, UNITS, &mt, &nt);
      const int batch = (int)((uint32_t)mt / (uint32_t)g.m_tiles_per_batch);
      const int mi0 = (int)((uint32_t)mt % (uint32_t)g.m_tiles_per_batch) * 2 * TBM + (int)rank * TBM;
      int64_t nrem = g.N - (int64_t)nt * TBN;
      const int n_mma = nrem >= TBN ? TBN : (int)((nrem + 15) & ~15LL);
      const int wrow = nt * TBN + (int)rank * (n_mma / 2);       // this CTA's half of the W rows of the tile
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait_cluster(BAR(PB_EMPTY + stage), phase ^ 1);
        if (lane == 0) trace_ev(g, 0, tr_i);
        ++tr_i;
        const uint32_t sb = stage0 + stage * P_STAGE_BYTES;
        const uint32_t wbar = mapa(BAR(PB_WFULL + stage), 0);
        const bool load_w = !WRES || cnt < (uint32_t)P_STAGES;        // W resident: first pass over the ring only
        if (elect_one()) {
          mbar_expect_tx(BAR(PB_AFULL + stage), TILE_BYTES);
          tma_load_3d(sb, &tmA, kb * TBK, mi0, batch, BAR(PB_AFULL + stage));
          if (load_w) {
            if (leader) mbar_expect_tx(BAR(PB_WFULL + stage), 4 * W_HALF_BYTES);   // hi and lo halves from the two CTAs
            tma_load_2d_pair(sb + TILE_BYTES, &tmWh, kb * TBK, wrow, wbar);
            tma_load_2d_pair(sb + TILE_BYTES + W_HALF_BYTES, &tmWl, kb * TBK, wrow, wbar);
          }
        }
        __syncwarp();
        ++cnt;
        if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    // Measured (tools/gemm_trace.py, K = 192, N-tile 128): the k-blocks of a tile complete 1300 / 600 / 1050 /
    // 790 / 800 / 790 clocks apart with the epilogue switched off (ideal 768 each: 12 MMAs x 64), i.e. ~800
    // clocks are lost at the start of every tile, and the epilogue's staging + store phase costs the third and
    // fourth k-block another ~1200.  Ruled out as the cause of the tile-start loss: an accumulator-switch
    // penalty of the tensor pipe (tools/probes/mma_probe.cu: none), the epilogue's tcgen05.ld traffic
    // (VASR_TC_DBG=3: same cadence), and this warp's own tile-boundary work (probing the barriers early and
    // hoisting the tile arithmetic took ~400 clocks off its path and changed nothing).
    if (leader) {
      uint32_t stage = 0, phase = 0, cnt = 0;     // cnt: k-steps issued so far (TMEM A slot = cnt % P_ASLOTS)
      uint32_t it = 0;
      int tr_i = 0;
      for (int64_t tile = first_tile; tile < total_tiles; tile += tile_stride, ++it) {
        MMA_TRACE(if (lane == 0) trace_ev(g, 10, (int)it);)
        int nt;
        int64_t mt_unused;
        tile_coords(g, tile, UNITS, &mt_unused, &nt);
        const int64_t nrem = g.N - (int64_t)nt * TBN;
        const uint32_t n_mma = nrem >= TBN ? (uint32_t)TBN : (uint32_t)((nrem + 15) & ~15LL);
        // M = 256 across the pair
        const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((n_mma >> 3) << 17) | ((256u >> 4) << 24);
        const uint32_t acc = it & 1u;
        mbar_wait_cluster(BAR(PB_TEMPTY + acc), ((it >> 1) & 1u) ^ 1u);
        tc_fence_after();
        MMA_TRACE(if (lane == 0) trace_ev(g, 11, (int)it);)
        const uint32_t tmem_d = tmem_base + acc * TBN;
#pragma unroll 1
        for (int kb = 0; kb < nkb; ++kb) {
          if (!WRES || cnt < (uint32_t)P_STAGES) mbar_wait_cluster(BAR(PB_WFULL + stage), phase);
          mbar_wait_cluster(BAR(PB_CONV + stage), phase);
          tc_fence_after();
          MMA_TRACE(if (lane == 0) trace_ev(g, 3, tr_i);)
          const uint32_t sb = stage0 + stage * P_STAGE_BYTES;
          const uint64_t db_hi = umma_desc(sb + TILE_BYTES), db_lo = umma_desc(sb + TILE_BYTES + W_HALF_BYTES);
          const uint32_t slot = cnt % P_ASLOTS;
          const uint32_t a_hi = tmem_base + TMEM_A0 + slot * 64, a_lo = a_hi + 32;
          if (elect_one()) {
#pragma unroll
            for (int k4 = 0; k4 < TBK / 8; ++k4) {
              const uint64_t adv = (uint64_t)(k4 * 2);
              umma_tf32_ts_pair(tmem_d, a_lo + 8 * k4, db_hi + adv, idesc, (kb | k4) != 0);
              umma_tf32_ts_pair(tmem_d, a_hi + 8 * k4, db_lo + adv, idesc, 1);
              umma_tf32_ts_pair(tmem_d, a_hi + 8 * k4, db_hi + adv, idesc, 1);
            }
            umma_commit_pair(BAR(PB_EMPTY + stage));
            umma_commit_pair(BAR(PB_AFREE + slot));
            if (kb == nkb - 1) umma_commit_pair(BAR(PB_TFULL + acc));
            MMA_TRACE(trace_ev(g, 4, tr_i);)
          }
          ++tr_i;
          ++cnt;
          __syncwarp();
          if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp < 6) {
    // ===================== converters (both CTAs): own A rows -> (hi, lo) -> own TMEM =====================
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + TMEM_A0;
    uint32_t stage = 0, phase = 0, cnt = 0, cit = 0;
    int tr_i = 0;
    for (int64_t tile = first_tile; tile < total_tiles; tile += tile_stride, ++cit) {
      // EPI_LNA: this thread sees its whole row of A go by; sum and sum of squares on the packed pipe, of the
      // values SHIFTED by the mean of the row's first 32 channels: E[x^2] - mean^2 cancels as (mean / std)^2, and a
      // common offset of 30 standard deviations on the rows cost four digits of the result without the shift
      // (measured on the CTC head: 2e-4 of the largest logit against 1.8e-6 for a plain fp32 LayerNorm + Linear).
      u64 sum2[2] = {0ull, 0ull}, sq2[2] = {0ull, 0ull}, shift2 = 0ull;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(BAR(PB_AFULL + stage), phase);
        if (threadIdx.x == 64) trace_ev(g, 1, tr_i);
        const uint8_t* arow = smem + stage * P_STAGE_BYTES + row * 128;
        if constexpr ((EPI & EPI_LNA) != 0) {
          if (kb == 0) {
            u64 s0 = 0ull, s1 = 0ull;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              const float4 v = *reinterpret_cast<const float4*>(arow + ((c ^ (row & 7)) << 4));
              s0 = add2(s0, pack2(v.x, v.y)); s1 = add2(s1, pack2(v.z, v.w));
            }
            const float shift = (hsum2(s0) + hsum2(s1)) * (1.0f / 32.0f);
            shift2 = pack2(-shift, -shift);
          }
        }
        uint32_t hi[32], lo[32];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          float4 v = *reinterpret_cast<const float4*>(arow + ((c ^ (row & 7)) << 4));
          if constexpr ((EPI & EPI_LNA) != 0) {
            // the SHIFTED row is what goes to the tensor core as well: acc = (x - shift) W'^T, so the epilogue's
            // correction is -(mean - shift) * rstd * s and nothing of the size of a common offset is left to cancel
            const u64 a = add2(pack2(v.x, v.y), shift2), b = add2(pack2(v.z, v.w), shift2);
            sum2[0] = add2(sum2[0], a); sum2[1] = add2(sum2[1], b);
            sq2[0] = fma2(a, a, sq2[0]); sq2[1] = fma2(b, b, sq2[1]);
            unpack2(a, v.x, v.y);
            unpack2(b, v.z, v.w);
          }
          hi[4 * c + 0] = rna_tf32(v.x); lo[4 * c + 0] = rna_tf32(v.x - __uint_as_float(hi[4 * c + 0]));
          hi[4 * c + 1] = rna_tf32(v.y); lo[4 * c + 1] = rna_tf32(v.y - __uint_as_float(hi[4 * c + 1]));
          hi[4 * c + 2] = rna_tf32(v.z); lo[4 * c + 2] = rna_tf32(v.z - __uint_as_float(hi[4 * c + 2]));
          hi[4 * c + 3] = rna_tf32(v.w); lo[4 * c + 3] = rna_tf32(v.w - __uint_as_float(hi[4 * c + 3]));
        }
        if constexpr ((EPI & EPI_LNA) != 0) {
          if (kb == nkb - 1) {
            // columns past K arrive as zeros (TMA fill) and add nothing.  The entry is written before this
            // warp's arrive on the conversion barrier of the tile's last k-block, which the tile's last MMAs,
            // their commit and the epilogue's wait for the accumulator all follow.
            const float inv = 1.0f / (float)g.K;
            if constexpr (SSTATS) {
              // rows past the end of A arrive as zeros: finite statistics that nobody uses
              const float dm = (hsum2(sum2[0]) + hsum2(sum2[1])) * inv;             // mean of the shifted row
              const float var = fmaxf(fmaf(-dm, dm, (hsum2(sq2[0]) + hsum2(sq2[1])) * inv), 0.f);
              const float rstd = 1.0f / sqrtf(var + g.ln_eps);
              sstats[(cit & 1u) * TBM + row] = make_float2(rstd, -dm * rstd);
            } else {
            int nt_unused;
            int64_t mt;
            tile_coords(g, tile, UNITS, &mt, &nt_unused);
            const uint32_t r = ((uint32_t)mt % (uint32_t)g.m_tiles_per_batch) * 2u * TBM + rank * TBM + (uint32_t)row;
            if (r < (uint32_t)g.rows_per_batch) {
              const float dm = (hsum2(sum2[0]) + hsum2(sum2[1])) * inv;
              const float var = fmaxf(fmaf(-dm, dm, (hsum2(sq2[0]) + hsum2(sq2[1])) * inv), 0.f);
              const float rstd = 1.0f / sqrtf(var + g.ln_eps);
              g.ln_stats[(int64_t)((uint32_t)mt / (uint32_t)g.m_tiles_per_batch) * g.rows_per_batch + r] =
                  make_float2(rstd, -dm * rstd);
            }
            }
          }
        }
        // the TMEM slot is free once the MMAs of its previous use (P_ASLOTS k-steps ago) have completed
        const uint32_t slot = cnt % P_ASLOTS;
        mbar_wait(BAR(PB_AFREE + slot), ((cnt / P_ASLOTS) & 1u) ^ 1u);
        tc_fence_after();
        tmem_st32(lane_addr + slot * 64, hi);
        tmem_st32(lane_addr + slot * 64 + 32, lo);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(mapa(BAR(PB_CONV + stage), 0));
        if (threadIdx.x == 64) trace_ev(g, 2, tr_i);
        ++tr_i;
        ++cnt;
        if (++stage == P_STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue (both CTAs): own 128 rows of the accumulator =====================
    if constexpr (TN == 192) {
      static_assert(TN != 192 || (ACT != ACT_SIGMOID && !PE && !QUANT), "192-column tiles: no pos-enc / quantised / sigmoid epilogue");
      epilogue_loop192<ACT, RESID, EPI>(g, smem + P_STAGES * P_STAGE_BYTES + (warp - 6) * EPI_STAGE_BYTES,
                              reinterpret_cast<float2*>(smem + Cfg::ROWFAC_OFFSET) + (warp - 6) * 32, sstats, warp, lane,
                              (uint32_t)first_tile, (uint32_t)tile_stride, (uint32_t)total_tiles, rank, BAR(PB_TFULL),
                              BAR(PB_TEMPTY));
    } else {
      static_assert(!(EPI & EPI_GATE), "the gate epilogue exists for 192-column tiles only");
      epilogue_loop<ACT, PE, RESID, QUANT, true, EPI>(g, smem + P_STAGES * P_STAGE_BYTES + (warp - 6) * EPI_STAGE_BYTES, warp, lane,
                                                 (uint32_t)first_tile, (uint32_t)tile_stride, (uint32_t)total_tiles, (uint32_t)UNITS, rank,
                                                 BAR(PB_TFULL), BAR(PB_TEMPTY), sstats);
    }
  }

  if (threadIdx.x == 6 * 32) trace_cta(g, 5);        // epilogue warp 6 done
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();           // nobody leaves while the peer may still signal or read it
  if (threadIdx.x == 0) trace_cta(g, 7);
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
  }
}

// w (n) -> hl[0..n) = rna_tf32(w), hl[n..2n) = rna_tf32(w - hi)
__global__ void __launch_bounds__(256) split_tf32_kernel(const float* __restrict__ w, float* __restrict__ hl,
                                                         int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const float x = w[i];
  const float h = __uint_as_float(rna_tf32(x));
  hl[i] = h;
  hl[n + i] = __uint_as_float(rna_tf32(x - h));
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

bool make_map(CUtensorMap* map, const float* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
              const uint32_t* box) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t gd[3], gs[2];
  cuuint32_t bx[3], es[3] = {1, 1, 1};
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<float*>(base), gd, gs, bx, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

}  // namespace

long long* g_trace = nullptr;   // set by vasr_debug_gemm_trace (tools/gemm_trace.py)
thread_local const TcVariant* tc_last_variant = nullptr;

namespace {
template <int FAMILY, int ACT, bool PE, bool RESID, bool QUANT, bool WRES = false, int TN = 128, int EPI = 0>
constexpr TcVariant kTcVariant = {FAMILY, TN, ACT, PE, RESID, QUANT, WRES, EPI};
}  // namespace

bool gemm_tc_supported(const GemmArgs& g) {
  if (!encode_fn()) return false;
  if (g.K % 4 != 0 || g.lda % 4 != 0 || g.batch_stride % 4 != 0) return false;
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  if (!al16(g.A) || !al16(g.W_split)) return false;
  // the epilogue moves 16-byte groups of four columns
  if ((g.N & 3) || (g.ldc & 3) || !al16(g.C) || (g.act_from & 3)) return false;
  if (g.bias && !al16(g.bias)) return false;
  if (g.q_scale && (!g.q_zp || !al16(g.q_scale) || !al16(g.q_zp))) return false;
  if (g.resid && ((g.ldr & 3) || !al16(g.resid))) return false;
  if (g.pe_time && ((g.pe_half & 3) || !al16(g.pe_time) || !al16(g.pe_freq))) return false;
  return true;
}

cudaError_t launch_split_tf32(const float* w, float* hl, int64_t n, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  split_tf32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(w, hl, n);
  return cudaGetLastError();
}

// Returns cudaErrorNotSupported when the tensor maps cannot be encoded (the caller then uses the
// CUDA-core kernel); any other error is a real launch failure.  g.W_split = [W_hi | W_lo].
cudaError_t launch_gemm_tc(const GemmArgs& g, int num_sms, cudaStream_t s, int64_t* launches) {
  if (g.M <= 0 || g.N <= 0) return cudaSuccess;
  if (!g.W_split || !gemm_tc_supported(g)) return cudaErrorNotSupported;
  const int64_t rpb = g.rows_per_batch > 0 ? g.rows_per_batch : g.M;
  const int64_t nb = g.rows_per_batch > 0 ? g.M / g.rows_per_batch : 1;
  if (nb * rpb != g.M) return cudaErrorNotSupported;
  if (g.pe_time && g.pe_rows != rpb) return cudaErrorNotSupported;   // pos-enc row == row within the batch
  const int64_t bstride = g.rows_per_batch > 0 ? g.batch_stride : rpb * g.lda;

  // CTA-pair kernel by default (4-7 % faster than the single-CTA one at config 2 once its cross-CTA barriers
  // stopped using cluster-scope acquire / release, which ptxas turns into CCTL.IVALL + MEMBAR.GPU);
  // the single-CTA kernel serves devices with one SM (and VASR_TC_PAIR=0 in a -DVASR_DEBUG build)
  static const bool use_pair = debug_env_int("VASR_TC_PAIR", 1) != 0;
  const bool pair = use_pair && num_sms >= 2;
  // 192-column tiles (PairCfg<192>).  VASR_TC_T192=0 turns them off.
  static const int t192_env = debug_env_int("VASR_TC_T192", 1);
  // Rule: 192-column tiles whenever N tiles into them without a tile narrower than 128 columns (192, 384, 512 =
  // 192 + 192 + 128, 576, 768, ...): a 128-column tile is exactly as fast as the control path (768 clocks of MMAs
  // per k-block against ~770), a 192-column one has 50 % more tensor work per k-block and per A tile loaded and
  // converted.  Measured against the 128-column tiling (W resident where it applied): in_proj -9 %, x / dt -6 %,
  // out_proj / ffn2 -18 %, fusion -17 %.  Instantiated for the plain (+ residual), softplus and GELU epilogues.
  // VASR_TC_T192=2 restricts it to the N that would otherwise end in a 64-column tile.
  // epilogue variants: folded LayerNorm (ln_s), argmax partials instead of the output (amax_val), gated fusion
  const bool lna = g.ln_s != nullptr, amax = g.amax_val != nullptr, gate = g.gate != 0;
  if (lna && (!pair || !g.ln_stats || g.K % TBK != 0 || g.K / TBK <= 4 || g.pe_time || g.resid || g.q_scale ||
              !(reinterpret_cast<uintptr_t>(g.ln_s) % 16 == 0) || !(g.act == ACT_NONE || (g.act == ACT_GELU && !amax))))
    return cudaErrorNotSupported;      // K / 32 > A slots: a row's entry is not rewritten before its tile's epilogue read it
  if (amax && (!pair || !g.amax_idx || g.act != ACT_NONE || g.pe_time || g.resid || g.q_scale || gate)) return cudaErrorNotSupported;
  if (gate && (!pair || lna || g.act != ACT_NONE || g.pe_time || g.resid || g.q_scale || g.N % 192 != 0)) return cudaErrorNotSupported;
  const bool inst192 = !g.pe_time && !g.q_scale && !amax && (!lna || g.act == ACT_GELU) &&
                       (g.act == ACT_NONE || ((g.act == ACT_SOFTPLUS || g.act == ACT_GELU) && !g.resid));
  const int64_t r192 = g.N % 192;
  bool t192 = pair && t192_env && inst192 && (r192 == 0 || r192 >= TBN);
  if (t192_env == 2 && g.N % TBN == 0) t192 = false;
  if (gate && !t192) return cudaErrorNotSupported;
  if (lna && g.act == ACT_GELU && !t192) return cudaErrorNotSupported;   // instantiated for the 192-column tiles only
  const int tn = t192 ? 192 : TBN;
  CUtensorMap tmA, tmWh, tmWl;
  {
    const uint64_t dims[3] = {(uint64_t)g.K, (uint64_t)rpb, (uint64_t)nb};
    const uint64_t str[2] = {(uint64_t)g.lda * 4, (uint64_t)(bstride > 0 ? bstride : g.lda) * 4};
    const uint32_t box[3] = {TBK, TBM, 1};
    if (!make_map(&tmA, g.A, 3, dims, str, box)) return cudaErrorNotSupported;
  }
  {
    const uint64_t dims[2] = {(uint64_t)g.K, (uint64_t)g.N};
    const uint64_t str[1] = {(uint64_t)g.K * 4};
    const uint32_t box[2] = {TBK, (uint32_t)(pair ? tn / 2 : tn)};       // a CTA of a pair loads half of the W tile
    if (!make_map(&tmWh, g.W_split, 2, dims, str, box)) return cudaErrorNotSupported;
    if (!make_map(&tmWl, g.W_split + g.N * g.K, 2, dims, str, box)) return cudaErrorNotSupported;
  }
  TcArgs a;
  a.M = g.M; a.N = g.N; a.K = g.K;
  a.rows_per_batch = rpb;
  a.n_batches = nb;
  a.m_tiles_per_batch = (int)((rpb + (pair ? 2 : 1) * TBM - 1) / ((pair ? 2 : 1) * TBM));
  a.n_tiles = (int)((g.N + tn - 1) / tn);
  a.C = g.C; a.ldc = g.ldc; a.bias = g.bias; a.act_from = g.act_from;
  a.q_scale = g.q_scale; a.q_zp = g.q_zp;
  a.resid = g.resid; a.ldr = g.ldr;
  a.pe_time = g.pe_time; a.pe_freq = g.pe_freq; a.pe_half = g.pe_half;
  a.ln_s = g.ln_s; a.ln_stats = reinterpret_cast<float2*>(g.ln_stats); a.ln_eps = g.ln_eps;
  a.amax_val = g.amax_val; a.amax_idx = g.amax_idx;
  a.trace = g_trace;
  static const int rot_env = debug_env_int("VASR_TC_ROT", 1);
  a.rotate_n = rot_env;
  static const int dbg_env = debug_env_int("VASR_TC_DBG", 0);
  a.dbg = dbg_env;
  static const int pf_env = debug_env_int("VASR_TC_PREFETCH", 0);   // measured: no gain
  a.prefetch = pf_env;

  const int64_t tiles = (int64_t)a.n_tiles * a.m_tiles_per_batch * nb;
  if (tiles >= (1LL << 31) || rpb >= (1LL << 31)) return cudaErrorNotSupported;
  const int64_t units = pair ? num_sms / 2 : num_sms;
  const unsigned grid = (unsigned)((tiles < units ? tiles : units) * (pair ? 2 : 1));
  // W resident (see TcArgs::wres): the k-blocks must tile the stage ring, every n-tile needs a pair, and each
  // pair should see enough m-tiles to amortise its private copy of W.  VASR_TC_WRES=0 turns it off.
  static const int wres_env = debug_env_int("VASR_TC_WRES", 1);
  a.wres = 0;
  if (pair && wres_env) {
    const int64_t nkb = (g.K + TBK - 1) / TBK, per = units / a.n_tiles, m_tiles = (int64_t)a.m_tiles_per_batch * nb;
    if (nkb <= P_STAGES && P_STAGES % nkb == 0 && per >= 1 && m_tiles >= 4 * per && (int64_t)grid == 2 * units) {
      a.wres = (int)per;
    }
  }
  const bool pe = g.pe_time != nullptr, rs = g.resid != nullptr;
  // W-resident instantiations exist for the plain and the GELU projection only (in_proj, ffn1, CTC head, q / k / v)
  if (pe || rs || g.q_scale || !(g.act == ACT_NONE || g.act == ACT_GELU) || t192) a.wres = 0;
  if (a.wres) a.rotate_n = 0;
  cudaError_t err = cudaSuccess;
  // each launch site names its instantiation once: VASR_GO1 / VASR_GO2 / VASR_GO192 (template arguments) launch it
  // and record it in tc_last_variant
  auto go1 = [&](auto kernel, const TcVariant* v) {
    tc_last_variant = v;
    err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (err == cudaSuccess) err = launch_k(kernel, dim3(grid), dim3(TC_THREADS), SMEM_BYTES, s, tmA, tmWh, tmWl, a);
  };
  auto go2 = [&](auto kernel, const TcVariant* v) {
    tc_last_variant = v;
    err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, P_SMEM_BYTES);
    if (err == cudaSuccess) err = launch_k(kernel, dim3(grid), dim3(TC_THREADS), P_SMEM_BYTES, s, tmA, tmWh, tmWl, a);
  };
  auto go192 = [&](auto kernel, const TcVariant* v) {
    tc_last_variant = v;
    err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PairCfg<192>::SMEM_BYTES);
    if (err == cudaSuccess)
      err = launch_k(kernel, dim3(grid), dim3(TC_THREADS), PairCfg<192>::SMEM_BYTES, s, tmA, tmWh, tmWl, a);
  };
#define VASR_GO1(...) go1(gemm_tc_kernel<__VA_ARGS__>, &kTcVariant<1, __VA_ARGS__>)
#define VASR_GO2(...) go2(gemm_tc2_kernel<__VA_ARGS__>, &kTcVariant<2, __VA_ARGS__>)
#define VASR_GO192(...) go192(gemm_tc2_kernel<__VA_ARGS__>, &kTcVariant<2, __VA_ARGS__>)
  if (t192) {
    a.rotate_n = 0;
    if (gate) VASR_GO192(ACT_NONE, false, false, false, false, 192, EPI_GATE);
    else if (lna) VASR_GO192(ACT_GELU, false, false, false, false, 192, EPI_LNA);
    else if (g.act == ACT_SOFTPLUS) VASR_GO192(ACT_SOFTPLUS, false, false, false, false, 192);
    else if (g.act == ACT_GELU) VASR_GO192(ACT_GELU, false, false, false, false, 192);
    else if (rs) VASR_GO192(ACT_NONE, false, true, false, false, 192);
    else VASR_GO192(ACT_NONE, false, false, false, false, 192);
    if (err != cudaSuccess) return err;
    if (launches) ++*launches;
    return cudaSuccess;
  }
  if (lna || amax) {      // plain projection with a folded LayerNorm and / or the argmax epilogue (CTC head, q, k | v)
    if (a.wres) {
      if (lna && amax) VASR_GO2(ACT_NONE, false, false, false, true, 128, EPI_LNA | EPI_AMAX);
      else if (lna) VASR_GO2(ACT_NONE, false, false, false, true, 128, EPI_LNA);
      else VASR_GO2(ACT_NONE, false, false, false, true, 128, EPI_AMAX);
    } else {
      if (lna && amax) VASR_GO2(ACT_NONE, false, false, false, false, 128, EPI_LNA | EPI_AMAX);
      else if (lna) VASR_GO2(ACT_NONE, false, false, false, false, 128, EPI_LNA);
      else VASR_GO2(ACT_NONE, false, false, false, false, 128, EPI_AMAX);
    }
    if (err != cudaSuccess) return err;
    if (launches) ++*launches;
    return cudaSuccess;
  }
  const bool quant = g.q_scale != nullptr;
  if (quant) {   // config 5: the quantised modules are plain projections, or the temporal-binding conv (GELU + pos-enc)
    if (rs || !((g.act == ACT_NONE && !pe) || (g.act == ACT_GELU && pe))) return cudaErrorNotSupported;
    if (pair) {
      if (pe) VASR_GO2(ACT_GELU, true, false, true);
      else VASR_GO2(ACT_NONE, false, false, true);
    } else {
      if (pe) VASR_GO1(ACT_GELU, true, false, true);
      else VASR_GO1(ACT_NONE, false, false, true);
    }
  }
#define VASR_TC_CASE(ACTV)                                                                   \
  if (!quant && g.act == ACTV) {                                                             \
    if (pair) {                                                                              \
      if (pe && rs) VASR_GO2(ACTV, true, true, false);                                       \
      else if (pe) VASR_GO2(ACTV, true, false, false);                                       \
      else if (rs) VASR_GO2(ACTV, false, true, false);                                       \
      else if (a.wres && ACTV == ACT_NONE) VASR_GO2(ACT_NONE, false, false, false, true);    \
      else if (a.wres && ACTV == ACT_GELU) VASR_GO2(ACT_GELU, false, false, false, true);    \
      else VASR_GO2(ACTV, false, false, false);                                              \
    } else {                                                                                 \
      if (pe && rs) VASR_GO1(ACTV, true, true, false);                                       \
      else if (pe) VASR_GO1(ACTV, true, false, false);                                       \
      else if (rs) VASR_GO1(ACTV, false, true, false);                                       \
      else VASR_GO1(ACTV, false, false, false);                                              \
    }                                                                                        \
  }
  VASR_TC_CASE(ACT_NONE)
  VASR_TC_CASE(ACT_GELU)
  VASR_TC_CASE(ACT_SOFTPLUS)
  VASR_TC_CASE(ACT_SIGMOID)
#undef VASR_TC_CASE
#undef VASR_GO1
#undef VASR_GO2
#undef VASR_GO192
  if (err != cudaSuccess) return err;
  if (launches) ++*launches;
  return cudaSuccess;
}

}  // namespace vasr
