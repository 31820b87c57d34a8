// Persistent LSTM recurrence (hidden 64, 1 layer, unidirectional) -- stereo_separator.py:37-43,107.
//
// The input projection X*W_ih^T + b_ih + b_hh is a tensor-core GEMM done by the conv engine
// (a k=1 conv, 128 -> 256); this kernel runs only the serial part:
//     g_t = xp_t + W_hh h_{t-1};  c_t = s(f) c_{t-1} + s(i) tanh(g);  h_t = s(o) tanh(c_t)
// One CTA of 256 threads owns S independent sequences for their whole length.  Thread
// (warp w, lane l) owns gate row  (l/8)*64 + 8w + (l%8)  -- its 64 W_hh weights stay in
// registers for the entire kernel -- so the four gates of hidden unit 8w+(l%8) sit in ONE
// warp and are combined with three warp shuffles; h_{t-1} is broadcast from shared memory
// (double buffered => a single block barrier per step).  Everything is fp32; only the copy of
// h that feeds the decoder convs is rounded to TF32.
#include "ar_common.cuh"
#include "pointwise.cuh"
#include "lstm_cell.cuh"

namespace ar {

// Packed 2-wide fp32 FMA (Blackwell FFMA2): halves the FMA issue slots of the 64-term dot product.
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

// offset (halves) of time step t inside one sequence of the time-blocked 256-channel pre-activation tensor
__device__ __forceinline__ long long tb_off(int t) {
  const int tr = HALO + t;
  return (long long)(tr >> 3) * (32 * 64) + (tr & 7) * 8;
}

// CAP: sequence b hands (h, c) to state_out[b] after local step cap[b] - 1 (cap[b] >= T: after the last step) and its
// scan continues.  A compile-time variant: the compare costs a share of the ~77-instruction step, so the scans without a
// per-sequence capture position keep the code they had.
template <int S, int PF, bool CAP = false>
__global__ void __launch_bounds__(256, (S <= 2) ? 2 : 1)
lstm_kernel(const __half* __restrict__ xp, long long xp_bs, int xp_Tp, const float* __restrict__ whh,
            __half* __restrict__ hout, long long h_bs, int h_Tp, int B, int T,
            const float* __restrict__ state_in, float* __restrict__ state_out, const int* __restrict__ cap = nullptr) {
  __shared__ __align__(16) float hbuf[2][S][LSTM_H];
  __shared__ __align__(16) float hstage[2][S][LSTM_BLK][LSTM_H];
  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int gate = lane >> 3;               // 0:i 1:f 2:g 3:o
  const int unit = warp * 8 + (lane & 7);
  const int row = gate * LSTM_H + unit;
  const int seq0 = blockIdx.x * S;

  unsigned long long w2[LSTM_H / 2];  // (w[2k], w[2k+1]) pairs
#pragma unroll
  for (int k = 0; k < LSTM_H; k += 4) {
    const float4 v = *reinterpret_cast<const float4*>(whh + row * LSTM_H + k);
    w2[k / 2] = pack2(v.x, v.y);
    w2[k / 2 + 1] = pack2(v.z, v.w);
  }

  float c[S];
  const __half* xrow[S];
  int capt[S];
#pragma unroll
  for (int s = 0; s < S; ++s) {
    const int b = min(seq0 + s, B - 1);  // surplus slots replay the last sequence, stores are masked
    if constexpr (CAP) capt[s] = seq0 + s < B ? min(cap[b], T) : 0;
    c[s] = 0.f;
    float h0 = 0.f;
    if (state_in != nullptr) {
      h0 = state_in[(long long)b * 2 * LSTM_H + unit];
      c[s] = state_in[(long long)b * 2 * LSTM_H + LSTM_H + unit];
    }
    if (gate == 0) hbuf[0][s][unit] = h0;
    const int xcol = unit * 4 + gate;   // pre-activation channels are stored [unit][gate], time-blocked (act_off_tb)
    xrow[s] = xp + (long long)b * xp_bs + (xcol >> 3) * 64 + (xcol & 7);
  }
  __syncthreads();

  // Pre-activations are prefetched PF steps ahead into a register set that is not live while the current
  // PF steps run (two sets, ping-pong over a 2*PF-step unrolled body), so the loads have PF steps to land
  // and never sit on the per-step critical path.
  float xa[S][PF], xb[S][PF];
#pragma unroll
  for (int s = 0; s < S; ++s)
#pragma unroll
    for (int k = 0; k < PF; ++k) xa[s][k] = __half2float(__ldg(xrow[s] + tb_off(min(k, T - 1))));

  int cur = 0;
  float hlast[S];
#pragma unroll
  for (int s = 0; s < S; ++s) hlast[s] = 0.f;

  auto run_block = [&](float (&xc)[S][PF], float (&xnext)[S][PF], int t0) {
#pragma unroll
    for (int s = 0; s < S; ++s)
#pragma unroll
      for (int k = 0; k < PF; ++k) xnext[s][k] = __half2float(__ldg(xrow[s] + tb_off(min(t0 + PF + k, T - 1))));
#pragma unroll
    for (int k = 0; k < PF; ++k) {
      const int t = t0 + k;
      if (t < T) {  // uniform across the block
        unsigned long long acc[S][4];
#pragma unroll
        for (int s = 0; s < S; ++s) {
          acc[s][0] = pack2(xc[s][k], 0.f);
          acc[s][1] = 0ull; acc[s][2] = 0ull; acc[s][3] = 0ull;
        }
#pragma unroll
        for (int j = 0; j < LSTM_H; j += 8) {
#pragma unroll
          for (int s = 0; s < S; ++s) {
            const ulonglong2 h0 = *reinterpret_cast<const ulonglong2*>(&hbuf[cur][s][j]);
            const ulonglong2 h1 = *reinterpret_cast<const ulonglong2*>(&hbuf[cur][s][j + 4]);
            acc[s][0] = fma2(w2[j / 2], h0.x, acc[s][0]);
            acc[s][1] = fma2(w2[j / 2 + 1], h0.y, acc[s][1]);
            acc[s][2] = fma2(w2[j / 2 + 2], h1.x, acc[s][2]);
            acc[s][3] = fma2(w2[j / 2 + 3], h1.y, acc[s][3]);
          }
        }
        const int sb = (t >> 3) & 1;
#pragma unroll
        for (int s = 0; s < S; ++s) {
          float a0, a1, a2, a3, a4, a5, a6, a7;
          unpack2(acc[s][0], a0, a1);
          unpack2(acc[s][1], a2, a3);
          unpack2(acc[s][2], a4, a5);
          unpack2(acc[s][3], a6, a7);
          const float pre = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
          const float a = (gate == 2) ? tanh_s(pre) : sigmoid_s(pre);
          const float af = __shfl_sync(0xffffffffu, a, (lane & 7) + 8);
          const float ag = __shfl_sync(0xffffffffu, a, (lane & 7) + 16);
          const float ao = __shfl_sync(0xffffffffu, a, (lane & 7) + 24);
          if (gate == 0) {
            c[s] = af * c[s] + a * ag;
            const float h = ao * tanh_f(c[s]);
            hlast[s] = h;
            hbuf[cur ^ 1][s][unit] = h;
            hstage[sb][s][t & 7][unit] = h;
            if constexpr (CAP) {
              if (t == capt[s] - 1) {
                state_out[(long long)(seq0 + s) * 2 * LSTM_H + unit] = h;
                state_out[(long long)(seq0 + s) * 2 * LSTM_H + LSTM_H + unit] = c[s];
              }
            }
          }
        }
        __syncthreads();
        cur ^= 1;
        if ((t & 7) == 7 || t == T - 1) {
          // flush up to 8 finished steps: [8 chunks][steps] x 16 bytes per sequence, coalesced along time
          const int tb = t & ~7;
          const int nst = t - tb + 1;
          for (int i = tid; i < S * 8 * LSTM_BLK; i += 256) {
            const int s = i / (8 * LSTM_BLK);
            const int ch = (i / LSTM_BLK) % 8;
            const int kk = i % LSTM_BLK;
            const int b = seq0 + s;
            if (b < B && kk < nst) {
              const float4 v0 = *reinterpret_cast<const float4*>(&hstage[sb][s][kk][8 * ch]);
              const float4 v1 = *reinterpret_cast<const float4*>(&hstage[sb][s][kk][8 * ch + 4]);
              const float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
              *reinterpret_cast<uint4*>(hout + act_off(h_bs, h_Tp, b, ch, tb + kk)) = pack_half8(v);
            }
          }
        }
      }
    }
  };

  for (int t0 = 0; t0 < T; t0 += 2 * PF) {
    run_block(xa, xb, t0);
    if (t0 + PF < T) run_block(xb, xa, t0 + PF);
  }
  if (!CAP && state_out != nullptr && gate == 0) {
#pragma unroll
    for (int s = 0; s < S; ++s) {
      const int b = seq0 + s;
      if (b < B) {
        state_out[(long long)b * 2 * LSTM_H + unit] = hlast[s];
        state_out[(long long)b * 2 * LSTM_H + LSTM_H + unit] = c[s];
      }
    }
  }
}

// ============================================================================ tensor-core recurrence
// Used when the batch exceeds two sequences per SM.  The recurrent mat-vec of a step becomes a [256 x 64] x [64 x 8]
// product on warp-level tensor-core MMAs (mma.sync m16n8k16, fp16 operands, fp32 accumulate).  W_hh is rounded to fp16
// like every other weight of the model and h is rounded to fp16 before it is fed back -- it is the same rounded value the
// decoder convs consume -- while the cell state c, the gate pre-activations and all gate math stay fp32 (tests: direct
// comparison with the fp32 oracle at 88 200 steps).
//
// A CTA owns NSEQ sequences and an SM holds two such CTAs, i.e. two independent recurrences to interleave: every step is
// one serial chain (h exchange -> MMAs -> gate functions -> barrier), and while one CTA sits in its barrier or its
// gate-function chain the other one issues.  The 8 recurrence warps own 8 hidden units each as two 16-row tiles, (i|f)
// and (g|o) of those units, so thread (gid, tig) finds all four gates of hidden unit 8w + gid for the sequences in MMA
// columns 2 tig and 2 tig + 1 in fixed accumulator registers -- no shuffles, no selects.
//   NSEQ = 4  (up to 8 sequences per SM): the eight MMA columns hold the sequences as (s0 s0 s1 s1 s2 s2 s3 s3); a thread
//             carries ONE cell (unit, sequence tig).  Shortest step: this is the latency-optimal shape.
//   NSEQ = 8  (more than 8 sequences per SM): eight distinct sequences; a thread carries TWO cells (unit, sequences 2 tig
//             and 2 tig + 1) whose gate-function chains interleave.  Same 8 MMAs per warp and step for twice the
//             sequences: at NSEQ = 4 the issue slots are 32 % busy and the step is a latency chain (ncu, round 1), so the
//             second cell rides in its shadow; the special-function unit (7 ex2 / rcp per cell) becomes the bound.
// h goes through shared memory ([seq][unit] fp16, padded stride: conflict-free 8-byte B-fragment loads).
//
// Warp specialisation: two extra "mover" warps do nothing but data movement -- they stage the next 8-step block of
// gate pre-activations (cp.async) and flush the previous block's hidden states -- so the eight recurrence warps run the
// bare step (5 LDS, 8 HMMA, the gate functions, 2 STS per cell) and meet at a named barrier of their own 256 threads.
// (With the flush inside the recurrence warps, the warp whose turn it was arrived ~40 instructions late at every step's
// barrier: 49.8 -> 43.4 ms per 1184-chunk step.)  The two groups meet once per 8-step block (named barrier 1, all 320
// threads): by then the movers have long finished.  The ping-pong index of the h exchange buffer is the step's parity
// inside the block -- a compile-time constant in the unrolled loop -- and full blocks run without the `step < T` tests.
constexpr int LM_HST = 68;      // padded [seq] row stride of the hidden-state staging buffer (floats): conflict-free stores

constexpr int LW_REC = 256;                        // recurrence warps
constexpr int LW_MOV = 64;                         // two mover warps
constexpr int LW_THREADS = LW_REC + LW_MOV;
template <int NSEQ>
struct LwGeom {
  static constexpr int XSTEP = NSEQ * LM_XS + 8;       // halves per staged step (+16 B: the 8 steps that consecutive lanes stage land in 8 bank groups)
  static constexpr int XBUF = LSTM_BLK * XSTEP;
  static constexpr int HSTEP = NSEQ * LM_HST + 4;      // floats per staged step of hidden states
  static constexpr int SMEM = 2 * XBUF * 2 + 2 * LSTM_BLK * HSTEP * 4 + 2 * NSEQ * LM_HS * 2;
};

template <int NSEQ, bool CAP = false>
__global__ void __launch_bounds__(LW_THREADS, 2)
lstm_mmaw_kernel(const __half* __restrict__ xp, long long xp_bs, int xp_Tp, const float* __restrict__ whh,
                 __half* __restrict__ hout, long long h_bs, int h_Tp, int B, int T,
                 const float* __restrict__ state_in, float* __restrict__ state_out, const int* __restrict__ cap = nullptr) {
  static_assert(NSEQ == 4 || NSEQ == 8, "four (duplicated columns) or eight sequences per CTA");
  using G = LwGeom<NSEQ>;
  constexpr int CELLS = NSEQ / 4;                              // cells per recurrence thread
  extern __shared__ __align__(16) float lm_smem[];
  __half* const xs = reinterpret_cast<__half*>(lm_smem);       // [2][8 steps][NSEQ][264] fp16 staged gate pre-activations
  float* const hstage = lm_smem + G::XBUF;                     // [2][8 steps][NSEQ][68] fp32
  __half* const hbuf = reinterpret_cast<__half*>(hstage + 2 * LSTM_BLK * G::HSTEP);   // [2][NSEQ][80] fp16
  const int tid = threadIdx.x;
  const int seq0 = blockIdx.x * NSEQ;
  const int nblk = (T + LSTM_BLK - 1) / LSTM_BLK;
  const int nfull = T / LSTM_BLK;

  if (tid >= LW_REC) {
    // ------------------------------------------------------------------ movers (warps 8, 9)
    const int ht = tid - LW_REC;
    const uint32_t xs_u32 = (uint32_t)__cvta_generic_to_shared(xs);
    auto stage_block = [&](int blk) {               // [NSEQ][32 chunks][8 steps] 16-byte pieces, 4 NSEQ per thread
      const int t0 = blk * LSTM_BLK;
      const uint32_t dst0 = xs_u32 + (uint32_t)((blk & 1) * G::XBUF * 2);
#pragma unroll 4
      for (int m = 0; m < 4 * NSEQ; ++m) {
        const int i = ht + LW_MOV * m;
        const int sq = i >> 8, piece = i & 255;
        const int ch = piece >> 3, k = piece & 7;
        const int b = min(seq0 + sq, B - 1);
        cp_async16(dst0 + (uint32_t)((k * G::XSTEP + sq * LM_XS + ch * 8) * 2), xp + act_off_tb(xp_bs, 32, b, ch, t0 + k));
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto flush_block = [&](int blk) {               // [NSEQ][8 chunks][8 steps] 16-byte items, NSEQ per thread
      const float* hst = hstage + (blk & 1) * (LSTM_BLK * G::HSTEP);
      const int t0 = blk * LSTM_BLK;
#pragma unroll
      for (int m = 0; m < NSEQ; ++m) {
        const int i = ht + LW_MOV * m;
        const int s = i >> 6, ch = (i >> 3) & 7, kk = i & 7;
        const int b = seq0 + s;
        if (b < B && t0 + kk < T) {
          const float* src = &hst[kk * G::HSTEP + s * LM_HST + 8 * ch];
          const float4 v0 = *reinterpret_cast<const float4*>(src);
          const float4 v1 = *reinterpret_cast<const float4*>(src + 4);
          const float v[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
          *reinterpret_cast<uint4*>(hout + act_off(h_bs, h_Tp, b, ch, t0 + kk)) = pack_half8(v);
        }
      }
    };
    stage_block(0);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    asm volatile("bar.sync 1, %0;" ::"n"(LW_THREADS) : "memory");
    for (int blk = 0; blk < nblk; ++blk) {
      if (blk + 1 < nblk) stage_block(blk + 1);
      if (blk > 0) flush_block(blk - 1);
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      asm volatile("bar.sync 1, %0;" ::"n"(LW_THREADS) : "memory");     // block blk is done, block blk + 1 has landed
    }
    flush_block(nblk - 1);
    return;
  }

  // -------------------------------------------------------------------- recurrence (warps 0..7)
  const int warp = tid >> 5, lane = tid & 31;
  const int gid = lane >> 2, tig = lane & 3;
  const int unit = warp * 8 + gid;
  uint32_t wfrag[2][4][4];
  load_whh_frags(whh, unit, tig, wfrag);
  const int upos = h_exchange_pos(unit);
  // this thread's cells: (unit, sequence tig * CELLS + j); the sequence of cell j sits in accumulator column 2 tig + j
  float c[CELLS], hl[CELLS];
  int capt[CELLS];
#pragma unroll
  for (int j = 0; j < CELLS; ++j) {
    const int seq = tig * CELLS + j;
    const int bq = min(seq0 + seq, B - 1);
    if constexpr (CAP) capt[j] = seq0 + seq < B ? min(cap[bq], T) : 0;
    c[j] = 0.f;
    hl[j] = 0.f;
    if (state_in != nullptr) {
      hl[j] = state_in[(long long)bq * 2 * LSTM_H + unit];
      c[j] = state_in[(long long)bq * 2 * LSTM_H + LSTM_H + unit];
    }
    hbuf[seq * LM_HS + upos] = __float2half_rn(hl[j]);
  }
  // B column gid = sequence gid (eight distinct) or gid / 2 (four, duplicated)
  const uint2* const hb_rd = reinterpret_cast<const uint2*>(hbuf + (NSEQ == 8 ? gid : gid >> 1) * LM_HS) + tig;
  __half* const hb_wr = hbuf + (tig * CELLS) * LM_HS + upos;
  const int xoff = (tig * CELLS) * LM_XS + unit * 4;          // [unit][i,f,g,o] of this thread's first cell inside a staged step
  const int hoff = (tig * CELLS) * LM_HST + unit;
  asm volatile("bar.sync 1, %0;" ::"n"(LW_THREADS) : "memory");

  // one step; `cur` (which half of hbuf holds h_{t-1}) is the step's parity inside the block: static when unrolled
  auto step = [&](const __half* xb, float* hst, int k) {
    const int cur = k & 1;
    uint2 q[CELLS];
#pragma unroll
    for (int j = 0; j < CELLS; ++j) q[j] = *reinterpret_cast<const uint2*>(xb + k * G::XSTEP + xoff + j * LM_XS);
    float acc[2][4];
#pragma unroll
    for (int tl = 0; tl < 2; ++tl)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[tl][i] = 0.f;
    const uint2* hb = hb_rd + cur * (NSEQ * LM_HS / 4);
#pragma unroll
    for (int kt = 0; kt < 4; ++kt) {
      const uint2 bf = hb[kt * 4];
      mma_f16_16x8x16(acc[0], wfrag[0][kt], bf.x, bf.y);
      mma_f16_16x8x16(acc[1], wfrag[1][kt], bf.x, bf.y);
    }
    if constexpr (CELLS == 2) {   // both cells of the thread through the packed 2-wide update (bit-identical to lstm_cell)
      float pi[2], pf[2], pg[2], po[2];
#pragma unroll
      for (int j = 0; j < 2; ++j) lstm_preact(acc[0][j], acc[0][2 + j], acc[1][j], acc[1][2 + j], q[j * (CELLS - 1)], pi[j], pf[j], pg[j], po[j]);
      lstm_cell2(pi[0], pi[1], pf[0], pf[1], pg[0], pg[1], po[0], po[1], c, hl);
    }
#pragma unroll
    for (int j = 0; j < CELLS; ++j) {
      if constexpr (CELLS != 2) {
        float pi, pf, pg, po;
        lstm_preact(acc[0][j], acc[0][2 + j], acc[1][j], acc[1][2 + j], q[j], pi, pf, pg, po);
        lstm_cell(pi, pf, pg, po, c[j], hl[j]);
      }
      hb_wr[(cur ^ 1) * (NSEQ * LM_HS) + j * LM_HS] = __float2half_rn(hl[j]);
      hst[k * G::HSTEP + hoff + j * LM_HST] = hl[j];
    }
  };
  auto capture = [&](int t) {                        // CAP: (h, c) of the cells whose capture step t is
#pragma unroll
    for (int j = 0; j < CELLS; ++j)
      if (t == capt[j] - 1) {
        const long long b = seq0 + tig * CELLS + j;
        state_out[b * 2 * LSTM_H + unit] = hl[j];
        state_out[b * 2 * LSTM_H + LSTM_H + unit] = c[j];
      }
  };
  for (int blk = 0; blk < nfull; ++blk) {
    const __half* xb = xs + (blk & 1) * G::XBUF;
    float* hst = hstage + (blk & 1) * (LSTM_BLK * G::HSTEP);
#pragma unroll
    for (int k = 0; k < LSTM_BLK; ++k) {
      step(xb, hst, k);
      if constexpr (CAP) capture(blk * LSTM_BLK + k);
      if (k < LSTM_BLK - 1) asm volatile("bar.sync 2, %0;" ::"n"(LW_REC) : "memory");
      else asm volatile("bar.sync 1, %0;" ::"n"(LW_THREADS) : "memory");
    }
  }
  if (nfull < nblk) {                                // ragged last block
    const __half* xb = xs + (nfull & 1) * G::XBUF;
    float* hst = hstage + (nfull & 1) * (LSTM_BLK * G::HSTEP);
    const int nst = T - nfull * LSTM_BLK;
#pragma unroll
    for (int k = 0; k < LSTM_BLK - 1; ++k) {
      if (k < nst) {   // uniform
        step(xb, hst, k);
        if constexpr (CAP) capture(nfull * LSTM_BLK + k);
        asm volatile("bar.sync 2, %0;" ::"n"(LW_REC) : "memory");
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(LW_THREADS) : "memory");
  }
  if (!CAP && state_out != nullptr) {
#pragma unroll
    for (int j = 0; j < CELLS; ++j) {
      const int b = seq0 + tig * CELLS + j;
      if (b < B) {
        state_out[(long long)b * 2 * LSTM_H + unit] = hl[j];
        state_out[(long long)b * 2 * LSTM_H + LSTM_H + unit] = c[j];
      }
    }
  }
}

template <int NSEQ, bool CAP>
static int launch_lstm_mmaw(const Act& xp, const float* whh, const Act& h_out, int B, int T, const float* state_in, float* state_out,
                            const int* cap, cudaStream_t stream) {
  static DeviceOnce attrs;
  if (attrs.pending()) {
    AR_CUDA_OK(cudaFuncSetAttribute(lstm_mmaw_kernel<NSEQ, CAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, LwGeom<NSEQ>::SMEM));
    // two CTAs (53 / 103 KB each) must fit: ask for the largest shared-memory carve-out, the driver's default heuristic sizes
    // it for ONE CTA and the second recurrence of the SM would run after the first instead of under it
    AR_CUDA_OK(cudaFuncSetAttribute(lstm_mmaw_kernel<NSEQ, CAP>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attrs.done();
  }
  lstm_mmaw_kernel<NSEQ, CAP><<<(B + NSEQ - 1) / NSEQ, LW_THREADS, LwGeom<NSEQ>::SMEM, stream>>>(
      xp.h(), xp.bs, xp.Tp, whh, h_out.h(), h_out.bs, h_out.Tp, B, T, state_in, state_out, cap);
  return AR_OK;
}

template <bool CAP>
static int launch_lstm_t(const Act& xp, const float* whh, const Act& h_out, int B, int T, const float* state_in, float* state_out,
                         const int* cap, cudaStream_t stream) {
  // One sequence per CTA on CUDA cores (two CTAs per SM) while that covers the batch; beyond two sequences per SM the
  // tensor-core kernel, two CTAs per SM: four sequences per CTA up to 8 per SM, eight per CTA beyond that.
  if (B > 8 * sm_count()) {
    AR_TRY((launch_lstm_mmaw<8, CAP>(xp, whh, h_out, B, T, state_in, state_out, cap, stream)));
  } else if (B > 2 * sm_count()) {
    AR_TRY((launch_lstm_mmaw<4, CAP>(xp, whh, h_out, B, T, state_in, state_out, cap, stream)));
  } else {
    lstm_kernel<1, 8, CAP><<<B, 256, 0, stream>>>(xp.h(), xp.bs, xp.Tp, whh, h_out.h(), h_out.bs, h_out.Tp, B, T, state_in,
                                                  state_out, cap);
  }
  return AR_OK;
}

int launch_lstm(const Act& xp, const float* whh, const Act& h_out, int B, int T, const float* state_in, float* state_out,
                const int* cap, cudaStream_t stream) {
  AR_CHECK(T >= 1 && B >= 1, AR_ERR_INVALID, "lstm: empty input");
  AR_CHECK(cap == nullptr || state_out != nullptr, AR_ERR_INVALID, "lstm: per-sequence capture needs state_out");
  if (cap != nullptr) {
    AR_TRY(launch_lstm_t<true>(xp, whh, h_out, B, T, state_in, state_out, cap, stream));
  } else {
    AR_TRY(launch_lstm_t<false>(xp, whh, h_out, B, T, state_in, state_out, nullptr, stream));
  }
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

}  // namespace ar
