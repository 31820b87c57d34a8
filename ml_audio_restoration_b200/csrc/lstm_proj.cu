// LSTM input projection + recurrence in ONE persistent kernel (stereo_separator.py:104-107; batches beyond 8 sequences per
// SM): the gate pre-activations  xp = W_ih x_t + b_ih + b_hh  never exist in HBM.
//
// Layer by layer the projection is the widest tensor of the whole chain -- 256 fp16 channels at 44.1 kHz, 45 MB per 2 s
// chunk, written by the encoder's last launch and read back by the scan: 1 KB of HBM traffic per time step and sequence
// (17 % of everything a chunk moves), the reason the encoder's last chain needs three accumulators in TMEM, and the tensor
// that bounds the chunk batch.  Here the scan kernel computes it itself, on the tensor pipe that the recurrence leaves
// idle: per block of 8 time steps ONE tcgen05 GEMM  D[128 x 256] = A[128 x 128] * W_ih^T  (rows = 8 steps x 16 sequences,
// fp16 operands from the encoder output e4b, fp32 accumulate in TMEM, two accumulators = all 512 columns), converted to
// the staged fp16 [step][sequence][unit][i,f,g,o] layout the recurrence warps already read.  The numbers are the ones the
// layer-by-layer path produces: same fp16 operands, fp32 accumulation, bias added in fp32, one rounding to fp16.
//
// One CTA per SM owns 16 sequences for their whole length:
//   warps  0 .. 15   recurrence: two independent groups of 8 warps x 8 sequences (lstm.cu's 8-sequence shape: mma.sync
//                    m16n8k16, W_hh fragments in registers, two cells per thread), each with its own named barrier per
//                    step -- while one group sits in its barrier or gate-function chain the other one issues
//   warps 16 .. 19   movers: (a) cp.async the next block's 128 x 128 operand rows (16-byte pieces: rows are step-major,
//                    a sequence's 8 steps are 128 contiguous bytes in HBM), (b) TMEM -> +bias -> fp16 -> staging buffer,
//                    (c) flush the previous block's hidden states to HBM.  Mover warp q owns TMEM lanes 32 q .. 32 q + 31
//                    = steps 2 q, 2 q + 1 of a block: the staging buffer is SINGLE (68 KB) and recycled per step pair --
//                    slot q is rewritten with the next block's steps as soon as both groups are past step 2 q + 1
//                    The last mover warp also issues the block's 8 tcgen05 MMAs (M 128, N 256, K 16; one elected thread)
//                    -- 20 warps = 640 threads leave 96 registers per thread, a 21st warp would cut that to 80.
// What it costs (ablation on a B200, 2368 sequences, ns per step): 581 with neither GEMM nor conversion, +85 for the movers'
// TMEM -> fp16 conversion, +150 for the GEMM -- the recurrence's mma.sync and the tcgen05 MMAs share the tensor pipe and
// shared-memory bandwidth (a 1-CTA N = 256 MMA reads 12 KB per K step), so HMMAs queue behind a block's 8 MMAs.  Pacing the
// K steps (clock spin in the mover), splitting N, and issuing them from a recurrence thread behind its own HMMAs were
// all measured and all slower; back-to-back issue by a mover warp is what is left.  Against lstm.cu's 8-sequence kernel
// on stored pre-activations the scan is ~17 % slower, the encoder's last launch 43 % faster (two GEMMs instead of three),
// the chain 3 % faster per 2368-chunk step, and a chunk's workspace peak no longer contains a 256-channel tensor.
// Shared memory: W_ih 64 KB (resident), operand rows 32 KB, staged pre-activations 68 KB, hidden-state staging 2 x 18 KB,
// h exchange 5 KB = 205 KB.
#include <cstring>
#include <vector>

#include "ar_common.cuh"
#include "pointwise.cuh"
#include "lstm_cell.cuh"
#include "umma_ptx.cuh"
#include "umma_epilogue.cuh"

namespace ar {

constexpr int LP_SEQ = 16;                       // sequences per CTA
constexpr int LP_REC = 512, LP_MOV = 128;        // recurrence / mover threads
constexpr int LP_THREADS = LP_REC + LP_MOV;
constexpr int LP_K = 128, LP_N = 256;
constexpr int LP_XSTEP = LP_SEQ * LM_XS + 8;     // halves per staged step
constexpr int LP_HS = 72;                        // padded [seq] row stride of the hidden-state staging buffer (halves)
constexpr int LP_HSTEP = LP_SEQ * LP_HS + 8;     // halves per staged step of hidden states
constexpr int LP_W_OFF = 0;
constexpr int LP_W_BYTES = (LP_K / 8) * LP_N * 16;            // [16 k-chunks][256 n][8] fp16
constexpr int LP_A_OFF = LP_W_OFF + LP_W_BYTES;
constexpr int LP_A_BYTES = (LP_K / 8) * 128 * 16;             // [16 k-chunks][128 rows][8] fp16
constexpr int LP_XS_OFF = LP_A_OFF + LP_A_BYTES;
constexpr int LP_XS_BYTES = LSTM_BLK * LP_XSTEP * 2;
constexpr int LP_HST_OFF = LP_XS_OFF + LP_XS_BYTES;
constexpr int LP_HST_BYTES = 2 * LSTM_BLK * LP_HSTEP * 2;
constexpr int LP_HB_OFF = LP_HST_OFF + LP_HST_BYTES;
constexpr int LP_HB_BYTES = 2 * LP_SEQ * LM_HS * 2;
constexpr int LP_BIAS_OFF = LP_HB_OFF + LP_HB_BYTES;
constexpr int LP_BAR_OFF = LP_BIAS_OFF + LP_N * 4;
constexpr int LP_SMEM = LP_BAR_OFF + 32 * 8;
static_assert(LP_XS_OFF % 16 == 0 && LP_HST_OFF % 16 == 0 && LP_HB_OFF % 16 == 0 && LP_BAR_OFF % 8 == 0, "alignment");
static_assert(LP_SMEM <= 227 * 1024, "shared memory");

struct LstmProjArgs {
  const __half* x;        // encoder output e4b, H8 [B][16][Tp][8]
  long long x_bs;
  int x_Tp;
  const __half* wih;      // packed B operand [16 k-chunks][256 n][8] fp16, n = unit * 4 + gate, rows pre-scaled
  const float* bias;      // [256] (b_ih + b_hh) pre-scaled, same order
  const float* whh;       // fp32 [256][64], rows pre-scaled, PyTorch gate-major order
  __half* hout;           // H8 [B][8][Tp][8]
  long long h_bs;
  int h_Tp;
  int B, T;
  const float* state_in;
  float* state_out;
  const int* cap;         // CAP: per-sequence capture step (lstm_kernel in lstm.cu)
};

template <bool CAP>
__global__ void __launch_bounds__(LP_THREADS, 1) lstm_proj_kernel(const __grid_constant__ LstmProjArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sbase = smem_u32(smem);
  __half* const xs = reinterpret_cast<__half*>(smem + LP_XS_OFF);
  __half* const hstage = reinterpret_cast<__half*>(smem + LP_HST_OFF);
  __half* const hbuf = reinterpret_cast<__half*>(smem + LP_HB_OFF);
  float* const s_bias = reinterpret_cast<float*>(smem + LP_BIAS_OFF);
  const uint32_t bar0 = sbase + LP_BAR_OFF;
  // mbarriers
  const uint32_t w_bar = bar0;
  const uint32_t a_full = bar0 + 8, a_empty = bar0 + 16;
  auto tfull = [&](int i) { return bar0 + 8u * (3 + i); };
  auto tempty = [&](int i) { return bar0 + 8u * (5 + i); };
  auto slot_full = [&](int q) { return bar0 + 8u * (7 + q); };
  auto slot_free = [&](int q) { return bar0 + 8u * (11 + q); };
  auto blk_done = [&](int i) { return bar0 + 8u * (15 + i); };
  auto hst_free = [&](int i) { return bar0 + 8u * (17 + i); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + LP_BAR_OFF + 8 * 20);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int seq0 = blockIdx.x * LP_SEQ;
  const int B = a.B, T = a.T;
  const int nblk = (T + LSTM_BLK - 1) / LSTM_BLK;

  if (tid == 0) {
    mbar_init(w_bar, 1);
    mbar_init(a_full, 4);
    mbar_init(a_empty, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(tfull(i), 1);
      mbar_init(tempty(i), 4);
      mbar_init(blk_done(i), 2);
      mbar_init(hst_free(i), 4);
    }
    for (int q = 0; q < 4; ++q) {
      mbar_init(slot_full(q), 1);
      mbar_init(slot_free(q), 2);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 16) tmem_alloc(smem_u32((const void*)tmem_slot), 512);
  for (int i = tid; i < LP_N; i += LP_THREADS) s_bias[i] = a.bias[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= 16) {
    // ------------------------------------------------------------------ movers
    const int q = warp - 16;                       // TMEM lane quarter == step pair of a block
    const int mt = tid - LP_REC;                   // 0 .. 127
    const uint32_t a_u32 = sbase + LP_A_OFF;
    // operand rows of block j: [16 seq][16 k-chunks][8 steps] 16-byte pieces.  Issued early, published (wait, proxy fence,
    // arrive) only just before the GEMM that reads them, so the copy's latency never stalls this warp.
    auto load_A = [&](int j) {
      if (j >= 1) mbar_wait(a_empty, (uint32_t)(j - 1) & 1u);
      const int t0 = j * LSTM_BLK;
      const int chunk = mt >> 3, step = mt & 7;
      const uint32_t dst = a_u32 + (uint32_t)(chunk * 2048 + step * 16 * 16);
#pragma unroll 4
      for (int sq = 0; sq < LP_SEQ; ++sq) {
        const int b = min(seq0 + sq, B - 1);
        cp_async16(dst + (uint32_t)(sq * 16), a.x + act_off(a.x_bs, a.x_Tp, b, chunk, t0 + step));
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto publish_A = [&]() {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      fence_async_smem();                          // generic-proxy (cp.async) writes -> visible to the tensor core's async proxy
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full);
    };
    auto convert = [&](int j) {                    // accumulator of block j -> staged fp16 pre-activations, slot q
      mbar_wait(tfull(j & 1), (uint32_t)(j >> 1) & 1u);
      if (j >= 1) mbar_wait(slot_free(q), (uint32_t)(j - 1) & 1u);
      tc_fence_after();
      const int step = 2 * q + (lane >> 4), sq = lane & 15;
      __half* const dst = xs + step * LP_XSTEP + sq * LM_XS;
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((j & 1) * LP_N);
      tmem_stream<32>(taddr, LP_N, [&](int cb, const uint32_t (&r)[32], int) {     // the next 32 columns load under this math
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const float4 b0 = *reinterpret_cast<const float4*>(s_bias + cb + 8 * v);
          const float4 b1 = *reinterpret_cast<const float4*>(s_bias + cb + 8 * v + 4);
          const float f[8] = {__uint_as_float(r[8 * v]) + b0.x,     __uint_as_float(r[8 * v + 1]) + b0.y,
                              __uint_as_float(r[8 * v + 2]) + b0.z, __uint_as_float(r[8 * v + 3]) + b0.w,
                              __uint_as_float(r[8 * v + 4]) + b1.x, __uint_as_float(r[8 * v + 5]) + b1.y,
                              __uint_as_float(r[8 * v + 6]) + b1.z, __uint_as_float(r[8 * v + 7]) + b1.w};
          *reinterpret_cast<uint4*>(dst + cb + 8 * v) = pack_half8(f);
        }
      });
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(tempty(j & 1));
        mbar_arrive(slot_full(q));
      }
    };
    auto flush = [&](int j) {                      // hidden states of block j: [16 seq][8 chunks][8 steps] 16-byte items
      mbar_wait(blk_done(j & 1), (uint32_t)(j >> 1) & 1u);
      const __half* hst = hstage + (j & 1) * (LSTM_BLK * LP_HSTEP);
      const int t0 = j * LSTM_BLK;
#pragma unroll
      for (int m = 0; m < 8; ++m) {
        const int i = mt + LP_MOV * m;
        const int s = i >> 6, ch = (i >> 3) & 7, kk = i & 7;
        const int b = seq0 + s;
        if (b < B && t0 + kk < T)
          *reinterpret_cast<uint4*>(a.hout + act_off(a.h_bs, a.h_Tp, b, ch, t0 + kk)) =
              *reinterpret_cast<const uint4*>(hst + kk * LP_HSTEP + s * LP_HS + 8 * ch);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(hst_free(j & 1));
    };
    // the block's GEMM, issued by one elected thread of the last mover warp once all four warps have staged the operand
    // rows (a_full) and drained the accumulator it overwrites (tempty)
    const uint32_t idesc = make_idesc_f16(128, LP_N);
    const uint64_t a_desc_hi = make_desc(0u, 128u * 16u, 128u);       // k-chunks 2 KB apart, 8-row groups 128 B apart
    const uint64_t b_desc_hi = make_desc(0u, (uint32_t)LP_N * 16u, 128u);
    auto issue = [&](int j) {
      if (q != 3) return;
      if (elect_one()) {
        mbar_wait(a_full, (uint32_t)j & 1u);
        if (j >= 2) mbar_wait(tempty(j & 1), (uint32_t)((j >> 1) - 1) & 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)((j & 1) * LP_N);
        uint32_t a_addr = (sbase + LP_A_OFF) >> 4, b_addr = (sbase + LP_W_OFF) >> 4;
#pragma unroll
        for (int kb = 0; kb < LP_K / 16; ++kb) {
          umma_f16(d_tmem, a_desc_hi | (uint64_t)a_addr, b_desc_hi | (uint64_t)b_addr, idesc, kb ? 1u : 0u);
          a_addr += 2 * 128;
          b_addr += 2 * LP_N;
        }
        umma_commit(a_empty);
        umma_commit(tfull(j & 1));
      }
      __syncwarp();
    };
    if (q == 3) {
      if (elect_one()) {
        mbar_expect_tx(w_bar, (uint32_t)LP_W_BYTES);
        for (int off = 0; off < LP_W_BYTES; off += 32768)
          bulk_g2s(sbase + LP_W_OFF + off, reinterpret_cast<const char*>(a.wih) + off, 32768u, w_bar);
        mbar_wait(w_bar, 0);
      }
      __syncwarp();
    }
    load_A(0);
    publish_A();
    issue(0);
    if (nblk > 1) {
      load_A(1);
      publish_A();
      issue(1);
    }
    // Per block j: convert FIRST (a warp's slot frees at step 2 q + 1 of block j - 1 and nothing else may delay it: with the
    // operand load in front, warp 0 sat behind warp 3's GEMM issue and the recurrence waited for slot 0 at every block
    // start, 10 % of its samples), then start the copy for block j + 2, flush block j - 1 once the recurrence is through
    // it, and only then publish the copy and issue GEMM j + 2 -- more than a block before its result is needed.
    for (int j = 0; j < nblk; ++j) {
      convert(j);
      if (j + 2 < nblk) load_A(j + 2);
      if (j >= 1) flush(j - 1);
      if (j + 2 < nblk) {
        publish_A();
        issue(j + 2);                       // accumulator j & 1 is drained once all four warps are through convert(j)
      }
    }
    flush(nblk - 1);
  } else {
    // ------------------------------------------------------------------ recurrence: group g = warps 8 g .. 8 g + 7, sequences 8 g .. 8 g + 7
    const int g = warp >> 3, wl = warp & 7;
    const int gid = lane >> 2, tig = lane & 3;
    const int unit = wl * 8 + gid;
    const bool g_lead = (tid & 255) == 0;
    uint32_t wfrag[2][4][4];
    load_whh_frags(a.whh, unit, tig, wfrag);
    const int upos = h_exchange_pos(unit);
    const int sl0 = g * 8 + tig * 2;               // this thread's cells: (unit, CTA-local sequences sl0, sl0 + 1)
    float c[2], hl[2];
    int capt[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int bq = min(seq0 + sl0 + j, B - 1);
      if constexpr (CAP) capt[j] = seq0 + sl0 + j < B ? min(a.cap[bq], T) : 0;
      c[j] = 0.f;
      hl[j] = 0.f;
      if (a.state_in != nullptr) {
        hl[j] = a.state_in[(long long)bq * 2 * LSTM_H + unit];
        c[j] = a.state_in[(long long)bq * 2 * LSTM_H + LSTM_H + unit];
      }
      hbuf[(sl0 + j) * LM_HS + upos] = __float2half_rn(hl[j]);
    }
    const uint2* const hb_rd = reinterpret_cast<const uint2*>(hbuf + (g * 8 + gid) * LM_HS) + tig;   // B column gid = sequence 8 g + gid
    __half* const hb_wr = hbuf + sl0 * LM_HS + upos;
    const int xoff = sl0 * LM_XS + unit * 4;       // [unit][i,f,g,o] of this thread's first cell inside a staged step
    const int hoff = sl0 * LP_HS + unit;
    if (g == 0) asm volatile("bar.sync 2, 256;" ::: "memory");
    else asm volatile("bar.sync 3, 256;" ::: "memory");

    auto step = [&](__half* hst, int k) {
      const int cur = k & 1;
      uint2 q[2];
#pragma unroll
      for (int j = 0; j < 2; ++j) q[j] = *reinterpret_cast<const uint2*>(xs + k * LP_XSTEP + xoff + j * LM_XS);
      float acc[2][4];
#pragma unroll
      for (int tl = 0; tl < 2; ++tl)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[tl][i] = 0.f;
      const uint2* hb = hb_rd + cur * (LP_SEQ * LM_HS / 4);
#pragma unroll
      for (int kt = 0; kt < 4; ++kt) {
        const uint2 bf = hb[kt * 4];
        mma_f16_16x8x16(acc[0], wfrag[0][kt], bf.x, bf.y);
        mma_f16_16x8x16(acc[1], wfrag[1][kt], bf.x, bf.y);
      }
      {
        float pi[2], pf[2], pg[2], po[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) lstm_preact(acc[0][j], acc[0][2 + j], acc[1][j], acc[1][2 + j], q[j], pi[j], pf[j], pg[j], po[j]);
        lstm_cell2(pi[0], pi[1], pf[0], pf[1], pg[0], pg[1], po[0], po[1], c, hl);
      }
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const __half hh = __float2half_rn(hl[j]);
        hb_wr[(cur ^ 1) * (LP_SEQ * LM_HS) + j * LM_HS] = hh;
        hst[k * LP_HSTEP + hoff + j * LP_HS] = hh;
      }
    };
    for (int blk = 0; blk < nblk; ++blk) {
      __half* hst = hstage + (blk & 1) * (LSTM_BLK * LP_HSTEP);
      const int nst = min(LSTM_BLK, T - blk * LSTM_BLK);
      if (blk >= 2) mbar_wait(hst_free(blk & 1), (uint32_t)((blk >> 1) - 1) & 1u);   // the movers have flushed block blk - 2
#pragma unroll
      for (int k = 0; k < LSTM_BLK; ++k) {
        if (k < nst) {   // uniform; always true except in a ragged last block
          if ((k & 1) == 0) mbar_wait(slot_full(k >> 1), (uint32_t)blk & 1u);
          step(hst, k);
          if constexpr (CAP) {
#pragma unroll
            for (int j = 0; j < 2; ++j)
              if (blk * LSTM_BLK + k == capt[j] - 1) {
                const long long b = seq0 + sl0 + j;
                a.state_out[b * 2 * LSTM_H + unit] = hl[j];
                a.state_out[b * 2 * LSTM_H + LSTM_H + unit] = c[j];
              }
          }
          if (g == 0) asm volatile("bar.sync 2, 256;" ::: "memory");
          else asm volatile("bar.sync 3, 256;" ::: "memory");
          if ((k & 1) && g_lead) mbar_arrive(slot_free(k >> 1));          // this group is past steps 2 q, 2 q + 1: slot q may be rewritten
        }
      }
      if (g_lead) mbar_arrive(blk_done(blk & 1));
    }
    if (!CAP && a.state_out != nullptr) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int b = seq0 + sl0 + j;
        if (b < B) {
          a.state_out[(long long)b * 2 * LSTM_H + unit] = hl[j];
          a.state_out[(long long)b * 2 * LSTM_H + LSTM_H + unit] = c[j];
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 16) tmem_dealloc(tmem_base, 512);
}

// W_ih^T as the K-major no-swizzle B operand of the projection GEMM: [16 k-chunks][256 n][8 k] fp16; `g` is the same
// 128 -> 256 GEMM (columns permuted to [unit][gate], rows pre-scaled) that the layer-by-layer path packs for the conv engine
void pack_lstm_proj(const float* G /* [128 cin][256 n] */, std::vector<uint16_t>& out) {
  out.assign((size_t)LP_K * LP_N, 0);
  for (int k = 0; k < LP_K; ++k)
    for (int n = 0; n < LP_N; ++n) {
      float v = G[(size_t)k * LP_N + n];
      if (v > HALF_MAX) v = HALF_MAX;
      if (v < -HALF_MAX) v = -HALF_MAX;
      const __half hv = __float2half_rn(v);
      uint16_t bits;
      memcpy(&bits, &hv, 2);
      out[((size_t)(k / 8) * LP_N + n) * 8 + (k % 8)] = bits;
    }
}

int launch_lstm_proj(const Act& x, const __half* wih_packed, const float* bias, const float* whh, const Act& h_out, int B, int T,
                     const float* state_in, float* state_out, const int* cap, cudaStream_t stream) {
  AR_CHECK(T >= 1 && B >= 1 && x.C == LP_K, AR_ERR_INVALID, "lstm_proj: bad input");
  AR_CHECK(cap == nullptr || state_out != nullptr, AR_ERR_INVALID, "lstm_proj: per-sequence capture needs state_out");
  static DeviceOnce attrs;
  if (attrs.pending()) {
    AR_CUDA_OK(cudaFuncSetAttribute(lstm_proj_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, LP_SMEM));
    AR_CUDA_OK(cudaFuncSetAttribute(lstm_proj_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LP_SMEM));
    attrs.done();
  }
  LstmProjArgs a;
  a.x = x.h(); a.x_bs = x.bs; a.x_Tp = x.Tp;
  a.wih = wih_packed; a.bias = bias; a.whh = whh;
  a.hout = h_out.h(); a.h_bs = h_out.bs; a.h_Tp = h_out.Tp;
  a.B = B; a.T = T; a.state_in = state_in; a.state_out = state_out; a.cap = cap;

  if (cap != nullptr) lstm_proj_kernel<true><<<(B + LP_SEQ - 1) / LP_SEQ, LP_THREADS, LP_SMEM, stream>>>(a);
  else lstm_proj_kernel<false><<<(B + LP_SEQ - 1) / LP_SEQ, LP_THREADS, LP_SMEM, stream>>>(a);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

}  // namespace ar
