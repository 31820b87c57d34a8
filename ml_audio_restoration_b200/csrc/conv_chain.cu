// Fused conv chains on the 2-CTA tcgen05 engine: a k-tap (dilated) Conv1d followed by one or two more convs, computed
// per 256-row tile pair WITHOUT writing the intermediate activations to HBM.  Three shapes of chain are instantiated:
//
//   (a) k3 dilated -> k1                 the StereoSeparator's `_dilated_block` (stereo_separator.py:49-64)
//   (b) k3 dilated -> k1 -> k1 (N = 256) the last block + the LSTM input projection behind it (stereo_separator.py:104-106)
//   (d) k7 -> k7                         two consecutive decoder layers of the StereoSeparator (stereo_separator.py:66-83:
//                                        128 -> 64 -> 32 per side), tile stride 122
//   (e) k5 -> k7 (one output column)     the super-resolution tail: hf_emphasis (k5 32 -> 32 + LeakyReLU) and the
//                                        reconstruction head (k7 32 -> 1) + linear x2 interpolation residual
//                                        (super_resolution.py:56-62, 92-99), tile stride 122, plain fp32 output
//   (c) k3 -> k3                         the U-Net's double conv (`_conv_block`, denoiser.py:51-60; max-pool copy fused) and
//                                        the super-resolution residual block (conv-BN-LReLU-conv-BN + skip,
//                                        super_resolution.py:104-122; the skip operand is the chain's own input)
//
//   G1: D1[256 x N1] (TMEM) = sum_taps A(rows from HBM via bulk copies, tap-shifted descriptors) * W1
//   E1: D1 -> +bias, LeakyReLU, fp16 -> shared memory, laid out as the K-major no-swizzle A operand of G2
//   G2: D2[256 x N2] = sum_taps2 I1(tap-shifted) * W2      (A straight from shared memory, W2 resident like W1)
//   E2: last stage: the usual fused epilogue to HBM (H8 or time-blocked; pool / residual);  otherwise -> I2 and G3 / E3.
//
// These layers are HBM-bound when run one by one (k1 128->128: 512 B of activation traffic per row for 32 K MACs; k3
// 32->32: 128 B per row for 3 K MACs), so removing the intermediate write + read removes 40-60 % of a block's traffic.
//
// (c): a k3 second stage needs one intermediate row on either side of its outputs, and an MMA produces exactly 128 rows,
// so a tile yields 126 outputs (tile stride S = 126): G1 computes the intermediate for times [t0 - 1, t0 + 127), G2 reads
// it with tap shifts 0 / 1 / 2 (two slack rows behind the buffer feed only the two masked output rows).  Intermediate rows
// whose time lies outside [0, T) are the second conv's ZERO PADDING, not conv-1 outputs: E1 writes zeros there.
//
// (b): TMEM holds 512 columns = 128 (G1) + 128 (G2) + 256 (G3), which leaves nothing to double-buffer -- and with single
// buffers a pipeline trace showed the tensor pipe idle while E1 drains G1's accumulator (period 6 030 cycles for 3 270
// cycles of MMAs).  G1 and G2 therefore ROTATE through the two 128-column buffers: tile t's G1 fills buffer t mod 2, E1
// drains it, the SAME buffer then takes tile t's G2 (E1 is done with it by the time I1 is complete), E2 drains it and
// hands it to G1 of tile t + 2.  G1 of tile t + 1 runs in the other buffer while tile t is in E1 / G2 / E2: G1's
// accumulator is effectively double-buffered without a column more.  (Running G3 as two N = 128 halves through one
// accumulator to free columns was measured first: E3 of the first half then sits between the halves, period 7 270.)
//
// Tile groups: with 32 / 64 output columns a tile is ~100 cycles of MMAs and ~150 cycles of epilogue work behind four mbarrier
// hand-overs of 400-900 cycles each (G1 -> E1 -> G2 -> E2; pipeline trace: 1 560 cycles per tile pair for the super-resolution
// block, 2.2 x what its HBM traffic needs).  Narrow k3 chains therefore move G = 2 or 4 CONSECUTIVE tiles per pipeline step:
// one contiguous run of (G - 1) S + R input rows per channel chunk, G accumulators per buffer in TMEM, G intermediate tiles
// per shared-memory buffer, one hand-over per group.
//
// Warp roles (every stage of the chain has its own issuer and its own epilogue group, so no warp ever waits for a
// result that depends on work it still has to issue):
//   warp 0            bulk-copy (TMA) producer: resident weights of all stages, then the activation ring of G1
//   warp 1 .. NG      issuer of GEMM g = warp-1 (leader CTA issues tcgen05.mma.cta_group::2; the peer's warp zero-pads
//                     its edge rows / forwards "my operand half is ready" arrivals to the leader)
//   then NG groups    epilogue group g drains the accumulator of GEMM g: to shared memory (g < NG-1) or to HBM (last)
#include "ar_common.cuh"
#include "umma_ptx.cuh"
#include "umma_epilogue.cuh"

namespace ar {

constexpr int CH_SMEM_BUDGET = 227 * 1024;
constexpr int CH_BAR_BYTES = 768;
constexpr int CH_BIAS_BYTES = 2048;      // <= 512 fp32 biases over all stages
constexpr int CH_MAX_STAGES = 16;
constexpr int CH_PREFETCH = 2;           // tile pairs the L2 prefetch runs ahead of the shared-memory ring

enum ChainEpi { CE_PLAIN = 0, CE_POOL = 1, CE_RES = 2, CE_HEAD = 3 };

// epilogue warps per stage
__host__ __device__ constexpr int ch_group_warps(int NG, int g) { return NG == 2 ? 8 : (g == 2 ? 8 : 4); }
__host__ __device__ constexpr int ch_threads(int NG) { return 32 * (1 + NG) + 32 * 16; }
__host__ __device__ constexpr int ch_maxreg(int NG) { return NG == 2 ? 104 : 96; }

struct ChainCfg {
  int kbs, stages, R, nks, stage_bytes;  // activation ring of the first GEMM
  int w_bytes[3], w_off[3];              // resident weight halves per CTA
  int i_off[2], i_bytes[2], nbI[2];      // intermediate operands (output of GEMM g = input of GEMM g+1)
  int RI;                                // rows of ONE TILE of an intermediate operand: 128 + (taps2 - 1)
  int G;                                 // tiles per group: a CTA works on G consecutive tiles per pipeline step (narrow k3 chains)
  int i_tile[2];                         // bytes of one tile of intermediate operand g (a buffer holds G of them)
  int acc_col[3], nbA[3], acc_n[3];      // TMEM columns: GEMM g buffer b, tile i at acc_col[g] + b * acc_n[g] + i * N[g]
  int tmem_cols;
  int stage_off, bar_off, bias_off, smem_bytes;
};

// Optional pipeline trace (ar_debug_chain_trace): CTA 0 records clock64() at pipeline events of its first
// CH_TRACE_TILES tile pairs; slots: 0/1 G1 issue begin/end, 2/3 G2 operands ready / issued, 4/5 E1 begin/end,
// 6/7 E_last begin/end, 8 first stage landed, 9 peer's first stage ready, 10/11 G3 ready / issued, 12/13 E2(mid) begin/end.
constexpr int CH_TRACE_TILES = 64;
__device__ __forceinline__ void trace_ev(long long* tr, int it, int ev) {
  if (tr != nullptr && blockIdx.x == 0 && it < CH_TRACE_TILES && (threadIdx.x & 31) == 0) tr[it * 16 + ev] = clock64();
}

__device__ __forceinline__ void trace_ev1(long long* tr, int it, int ev) {   // caller is a single elected thread
  if (tr != nullptr && blockIdx.x == 0 && it < CH_TRACE_TILES) tr[it * 16 + ev] = clock64();
}

// buffer index / mbarrier phase of the u-th use of a set of nb (1 or 2) buffers
constexpr int CH_MAX_BUF = 2;
__device__ __forceinline__ int buf_of(int u, int nb) { return u & (nb - 1); }
__device__ __forceinline__ uint32_t phase_of(int u, int nb) { return (uint32_t)(u >> (nb >> 1)) & 1u; }   // nb >> 1 == log2(nb) for 1, 2

// GRP: compiled with tile groups (cfg.G tiles per pipeline step, narrow k3 chains); false pins G = 1 at compile time so the
// wide chains keep their register allocation
template <int TAPS, int NG, int TAPS2, int EPI, bool GRP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(ch_threads(NG), 1) __maxnreg__(ch_maxreg(NG))
conv_chain_kernel(const __grid_constant__ ChainParams cp, const __grid_constant__ ChainCfg cfg, int num_pairs) {
  static_assert(!GRP || (NG == 2 && (TAPS == 3 || TAPS == 5)), "tile groups are for the narrow two-GEMM k3 / k5 chains");
  static_assert(TAPS2 == 1 || NG == 2, "a k-tap second stage is a two-GEMM chain");
  static_assert(EPI == CE_PLAIN || NG == 2, "pool / residual / head epilogues belong to the two-GEMM chains");
  constexpr int S = TILE_M - (TAPS2 - 1);          // tile stride = outputs per tile
  constexpr int LEAD = (TAPS2 - 1) / 2;            // intermediate row r of a tile is time  tile * S - LEAD + r
  constexpr bool ROTATE = NG == 3;                 // G1 and G2 share two rotating accumulator buffers (see (b) above)
  extern __shared__ __align__(1024) uint8_t smem[];
  const ConvParams& p = cp.p;
  const uint32_t sbase = smem_u32(smem);
  const uint32_t stage_base = sbase + cfg.stage_off;
  uint8_t* const stage_ptr = smem + cfg.stage_off;
  const uint32_t bar_base = sbase + cfg.bar_off;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (CH_MAX_STAGES + s); };
  constexpr int B0 = 3 * CH_MAX_STAGES;
  auto tfull_bar = [&](int g, int b) { return bar_base + 8u * (B0 + g * CH_MAX_BUF + b); };
  auto tempty_bar = [&](int g, int b) { return bar_base + 8u * (B0 + 3 * CH_MAX_BUF + g * CH_MAX_BUF + b); };      // leader only
  auto ifull_bar = [&](int g, int b) { return bar_base + 8u * (B0 + 6 * CH_MAX_BUF + g * CH_MAX_BUF + b); };       // leader only: epilogue group g of BOTH CTAs -> issuer g+1
  auto iempty_bar = [&](int g, int b) { return bar_base + 8u * (B0 + 8 * CH_MAX_BUF + g * CH_MAX_BUF + b); };
  const uint32_t w_bar = bar_base + 8u * (B0 + 10 * CH_MAX_BUF);
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + cfg.bar_off + 8 * (B0 + 10 * CH_MAX_BUF + 1));
  static_assert(8 * (B0 + 10 * CH_MAX_BUF + 2) <= CH_BAR_BYTES, "barrier block too small");
  float* const s_bias = reinterpret_cast<float*>(smem + cfg.bias_off);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < cfg.stages; ++s) {
      // the leader's "stage full" also collects the peer's "my rows have landed" arrive: one wait per stage for the issuer
      mbar_init(full_bar(s), leader ? 2 : 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int g = 0; g < NG; ++g)
      for (int b = 0; b < CH_MAX_BUF; ++b) {
        mbar_init(tfull_bar(g, b), 1);
        mbar_init(tempty_bar(g, b), 2 * ch_group_warps(NG, g));
      }
    for (int g = 0; g < NG - 1; ++g)
      for (int b = 0; b < CH_MAX_BUF; ++b) {
        mbar_init(ifull_bar(g, b), 2 * ch_group_warps(NG, g));
        mbar_init(iempty_bar(g, b), 1);
      }
    mbar_init(w_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc2(smem_u32((const void*)tmem_slot), (uint32_t)cfg.tmem_cols);
  {
    int off = 0;
    for (int g = 0; g < NG; ++g) {
      for (int i = threadIdx.x; i < cp.N[g]; i += blockDim.x) s_bias[off + i] = cp.bias[g][i];
      off += cp.N[g];
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int tpi = p.tiles_per_item;                // tiles (of S output rows) per batch item
  const int G = GRP ? cfg.G : 1;                   // tiles per group
  const int gpi = (tpi + G - 1) / G;               // groups per batch item
  const int ppi = (gpi + 1) >> 1;                  // group pairs per batch item
  const int R = cfg.R;                             // input rows of a group's run: (G - 1) S + 128 + (taps - 1) dil
  const int RI = cfg.RI;
  const int pair0 = blockIdx.x >> 1;
  const int pair_step = gridDim.x >> 1;
  const int n_local = pair0 < num_pairs ? (num_pairs - pair0 + pair_step - 1) / pair_step : 0;   // group pairs of this cluster
  // this CTA's group of pair pi of an item, and the first input row (time index) of its run: group * G * S - LEAD - pad_left;
  // an idle half (odd group count) re-reads the item's last group, whose rows then get zeroed
  auto group_of = [&](int pi) { return pi * 2 + (int)rank; };
  auto run_t0 = [&](int pi) {
    int gl = group_of(pi);
    if (gl > gpi - 1) gl = gpi - 1;
    return gl * G * S - LEAD - p.pad_left;
  };
  // rows of the run that exist in the padded buffer (the last group may reach past it)
  auto run_rows = [&](int t0) {
    const int avail = p.in_Tp - (HALO + t0);
    return R < avail ? R : avail;
  };

  if (warp == 0) {
    // ------------------------------------------------------------------ producer: resident weights, then the activation ring
    if (elect_one()) {
      uint32_t total = 0;
      for (int g = 0; g < NG; ++g) total += (uint32_t)cfg.w_bytes[g];
      mbar_expect_tx(w_bar, total);
      for (int g = 0; g < NG; ++g) {
        const char* wsrc = reinterpret_cast<const char*>(cp.w[g]) + (size_t)rank * cfg.w_bytes[g];
        for (int off = 0; off < cfg.w_bytes[g]; off += 32768) {
          const int n = cfg.w_bytes[g] - off < 32768 ? cfg.w_bytes[g] - off : 32768;
          bulk_g2s(sbase + cfg.w_off[g] + off, wsrc + off, (uint32_t)n, w_bar);
        }
      }
      int s = 0;
      uint32_t ph = 0;
      const uint32_t pitch = (uint32_t)(R * 16);                 // shared-memory distance between 8-channel chunks of a stage
      const long long chunk_stride = (long long)p.in_Tp * 8;
      const int chunks_per_stage = cfg.kbs * 2;
      PairIter pit(pair0, pair_step, ppi), pre(pair0, pair_step, ppi);
      const int n_chunks = p.Cin >> 3;
      // L2 prefetch runs CH_PREFETCH tile pairs ahead of the ring
      const int pre_dist = CH_PREFETCH;
      for (int d = 0; d < pre_dist && d < n_local; ++d, pre.next()) {
        const int t0 = run_t0(pre.pi);
        const __half* ps = p.in + act_off(p.in_bs, p.in_Tp, pre.b, p.in_coff8, t0);
        const uint32_t nb = (uint32_t)(run_rows(t0) * 16);
        for (int c = 0; c < n_chunks; ++c, ps += chunk_stride) bulk_prefetch_l2(ps, nb);
      }
      for (int it = 0; it < n_local; ++it, pit.next()) {
        const int t0 = run_t0(pit.pi);
        const __half* src = p.in + act_off(p.in_bs, p.in_Tp, pit.b, p.in_coff8, t0);
        const uint32_t row_bytes = (uint32_t)(run_rows(t0) * 16);
        const bool do_pre = it + pre_dist < n_local;
        const __half* ps = nullptr;
        uint32_t pre_bytes = 0;
        if (do_pre) {
          const int tp = run_t0(pre.pi);
          ps = p.in + act_off(p.in_bs, p.in_Tp, pre.b, p.in_coff8, tp);
          pre_bytes = (uint32_t)(run_rows(tp) * 16);
          pre.next();
        }
        for (int ks = 0; ks < cfg.nks; ++ks) {
          const uint32_t fb = full_bar(s);
          mbar_wait(empty_bar(s), ph ^ 1u);
          mbar_expect_tx(fb, (uint32_t)chunks_per_stage * row_bytes);
          uint32_t dst = stage_base + s * cfg.stage_bytes;
          for (int c = 0; c < chunks_per_stage; ++c) {
            bulk_g2s(dst, src, row_bytes, fb);
            if (do_pre) { bulk_prefetch_l2(ps, pre_bytes); ps += chunk_stride; }
            dst += pitch;
            src += chunk_stride;
          }
          if (++s == cfg.stages) { s = 0; ph ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ issuer of G1: k-tap conv, rows streamed through the ring.
    // ONE elected thread walks the loop (waits, rare edge zero-fill, MMA issue, commits).
    if (elect_one()) {
      mbar_wait(w_bar, 0);
      int s = 0;
      uint32_t ph = 0;
      const int N1 = cp.N[0], Nh = N1 >> 1;
      const uint32_t idesc = make_idesc_f16(256, N1);
      const uint64_t a_desc_hi = make_desc(0u, (uint32_t)(R * 16), 128u);
      const uint64_t b_desc_hi = make_desc(0u, (uint32_t)(Nh * 16), 128u);
      const uint32_t b_step = (uint32_t)(Nh * 2);
      const uint32_t a_step = (uint32_t)(2 * R);
      const uint32_t dil_u = (uint32_t)p.dil;
      const uint32_t w_addr0 = (sbase + cfg.w_off[0]) >> 4;
      const int nbA = cfg.nbA[0];
      const uint32_t full0_leader = mapa_u32(full_bar(0), 0);
      PairIter pit(pair0, pair_step, ppi);
      for (int it = 0; it < n_local; ++it, pit.next()) {
        const int tfirst = run_t0(pit.pi);
        const bool dead = group_of(pit.pi) > gpi - 1;          // no such group: contribute zeros
        const bool edge = dead || (tfirst < 0) || (tfirst + R > p.Tin);
        const int buf = buf_of(it, nbA);
        if (leader) {
          // buffer free: drained by E1 of its previous G1 -- or, rotating, by E2 of the G2 that ran in it after that
          mbar_wait(tempty_bar(ROTATE ? 1 : 0, buf), phase_of(it, nbA) ^ 1u);
          tc_fence_after();
        }
        trace_ev1(cp.trace, it, 0);
        const uint32_t d_tmem0 = tmem_base + (uint32_t)(cfg.acc_col[0] + buf * cfg.acc_n[0]);
        uint32_t b_addr = w_addr0;
        for (int ks = 0; ks < cfg.nks; ++ks) {
          mbar_wait(full_bar(s), ph);                          // leader: own rows landed AND the peer's arrive
          if (ks == 0) trace_ev1(cp.trace, it, 8);
          if (edge) {  // conv zero padding of this CTA's rows (first / last groups of an item only), incl. rows never loaded
            uint8_t* a_ptr = stage_ptr + s * cfg.stage_bytes;
            const int r_lo = dead ? R : (tfirst < 0 ? -tfirst : 0);                 // rows [0, r_lo) lie before the signal
            const int r_hi = dead ? R : (p.Tin - tfirst < R ? p.Tin - tfirst : R);  // rows [r_hi, R) behind it
            for (int c = 0; c < cfg.kbs * 2; ++c) {
              for (int r = 0; r < r_lo; ++r) *reinterpret_cast<float4*>(a_ptr + (c * R + r) * 16) = make_float4(0.f, 0.f, 0.f, 0.f);
              for (int r = r_hi < 0 ? 0 : r_hi; r < R; ++r) *reinterpret_cast<float4*>(a_ptr + (c * R + r) * 16) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
            fence_async_smem();
          }
          if (!leader) {
            if (edge) mbar_arrive_remote_release(full0_leader + 8u * s);   // zero-padding writes must be visible
            else mbar_arrive_remote(full0_leader + 8u * s);
          } else {
            const uint32_t a_stage = (stage_base + s * cfg.stage_bytes) >> 4;
            for (int i = 0; i < G; ++i) {                      // the tiles of the group: same stage, rows shifted by i * S
              uint32_t a_addr = a_stage + (uint32_t)(i * S);
              uint32_t bw = b_addr;
              const uint32_t d_tmem = d_tmem0 + (uint32_t)(i * N1);
              for (int kb = 0; kb < cfg.kbs; ++kb) {
#pragma unroll
                for (int j = 0; j < TAPS; ++j)
                  umma2_f16(d_tmem, a_desc_hi | (uint64_t)(a_addr + (uint32_t)j * dil_u),
                            b_desc_hi | (uint64_t)(bw + (uint32_t)j * b_step), idesc, (ks | kb | j) ? 1u : 0u);
                bw += (uint32_t)TAPS * b_step;
                a_addr += a_step;
              }
            }
            b_addr += (uint32_t)(cfg.kbs * TAPS) * b_step;
            umma_commit2(empty_bar(s));
            if (ks == cfg.nks - 1) umma_commit2(tfull_bar(0, buf));
          }
          if (++s == cfg.stages) { s = 0; ph ^= 1u; }
        }
        trace_ev1(cp.trace, it, 1);
      }
    }
    __syncwarp();
  } else if (warp <= NG) {
    // ------------------------------------------------------------------ issuer of GEMM g >= 1: A = operand written by epilogue group g-1
    const int g = warp - 1;
    mbar_wait(w_bar, 0);
    const int K = cp.N[g - 1], Ng = cp.N[g], Nh = Ng >> 1;
    const int nbI = cfg.nbI[g - 1], nbA = cfg.nbA[g];
    const uint32_t idesc = make_idesc_f16(256, Ng);
    const uint64_t a_desc_hi = make_desc(0u, (uint32_t)(RI * 16), 128u);
    const uint64_t b_desc_hi = make_desc(0u, (uint32_t)(Nh * 16), 128u);
    const uint32_t b_step = (uint32_t)(Nh * 2);
    const uint32_t w_addr0 = (sbase + cfg.w_off[g]) >> 4;
    const int taps_g = (g == 1) ? TAPS2 : 1;
    // Only the leader issues.  The operand rows each CTA wrote for itself are published by its epilogue warps
    // (fence.proxy.async, then an arrive on the LEADER's barrier -- same relaxed remote arrive as the per-stage
    // "my half is in place" handshake of G1: the data is read by the writer's own SM, only the trigger is remote).
    if (leader && elect_one()) {
      for (int it = 0; it < n_local; ++it) {
        const int bi = buf_of(it, nbI);
        mbar_wait(ifull_bar(g - 1, bi), phase_of(it, nbI));   // both CTAs' operand rows are in their shared memory
        const int buf = buf_of(it, nbA);
        // accumulator free?  Rotating G2: it is the buffer E1 of this very tile just drained (implied by ifull above)
        if (!(ROTATE && g == 1)) mbar_wait(tempty_bar(g, buf), phase_of(it, nbA) ^ 1u);
        tc_fence_after();
        trace_ev1(cp.trace, it, g == 1 ? 2 : 10);
        for (int i = 0; i < G; ++i) {
          const uint32_t d_tmem = tmem_base + (uint32_t)(cfg.acc_col[g] + buf * cfg.acc_n[g] + i * Ng);
          uint32_t a_addr = (sbase + cfg.i_off[g - 1] + bi * cfg.i_bytes[g - 1] + i * cfg.i_tile[g - 1]) >> 4;
          uint32_t b_addr = w_addr0;
          for (int kb = 0; kb < K / 16; ++kb) {
            if (NG == 2) {                                     // the second GEMM of a two-GEMM chain: taps known at compile time
#pragma unroll
              for (int j = 0; j < TAPS2; ++j)
                umma2_f16(d_tmem, a_desc_hi | (uint64_t)(a_addr + (uint32_t)j), b_desc_hi | (uint64_t)(b_addr + (uint32_t)j * b_step), idesc,
                          (kb | j) ? 1u : 0u);
            } else {
              for (int j = 0; j < taps_g; ++j)
                umma2_f16(d_tmem, a_desc_hi | (uint64_t)(a_addr + (uint32_t)j), b_desc_hi | (uint64_t)(b_addr + (uint32_t)j * b_step), idesc,
                          (kb | j) ? 1u : 0u);
            }
            a_addr += (uint32_t)(2 * RI);
            b_addr += (uint32_t)taps_g * b_step;
          }
        }
        umma_commit2(iempty_bar(g - 1, bi));                // both CTAs may overwrite this operand buffer
        umma_commit2(tfull_bar(g, buf));
        trace_ev1(cp.trace, it, g == 1 ? 3 : 11);
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ epilogue groups: own 128 rows of one stage's accumulator
    int g = 0, w0 = 1 + NG;
    while (g < NG - 1 && warp >= w0 + ch_group_warps(NG, g)) { w0 += ch_group_warps(NG, g); ++g; }
    const int gw = ch_group_warps(NG, g);
    const int q = warp & 3;                                  // TMEM lane quarter this warp may read
    const int part = (warp - w0) >> 2, nparts = gw >> 2;     // column part
    const int Ng = cp.N[g];
    const int wcols = Ng / nparts < 16 ? 16 : Ng / nparts;
    const int col_lo = part * wcols;                         // first accumulator column (= output channel) of this warp
    const bool active = col_lo < Ng;
    const float slope = cp.lrelu[g] ? LRELU_SLOPE : 1.0f;
    int bias_off = 0;
    for (int i = 0; i < g; ++i) bias_off += cp.N[i];
    const int nbA = cfg.nbA[g];
    const uint32_t tempty0_leader = mapa_u32(tempty_bar(g, 0), 0);
    const uint32_t taddr0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(cfg.acc_col[g] + col_lo);
    const bool tracer = (warp == w0);
    if (g < NG - 1) {
      // accumulator -> bias, LeakyReLU, fp16 -> this CTA's operand rows of GEMM g+1
      const float* bw = s_bias + bias_off + col_lo;
      const float ca = 0.5f * (1.0f + slope), cbk = 0.5f * (1.0f - slope);
      const int nbI = cfg.nbI[g];
      const uint32_t ifull0_leader = mapa_u32(ifull_bar(g, 0), 0);
      PairIter pit(pair0, pair_step, ppi);
      for (int it = 0; it < n_local; ++it, pit.next()) {
        const int buf = buf_of(it, nbA);
        const int bi = buf_of(it, nbI);
        mbar_wait(tfull_bar(g, buf), phase_of(it, nbA));
        mbar_wait(iempty_bar(g, bi), phase_of(it, nbI) ^ 1u);   // GEMM g+1 of the previous user has read the buffer
        tc_fence_after();
        if (tracer) trace_ev(cp.trace, it, g == 0 ? 4 : 12);
        const int gl = group_of(pit.pi);
        // a k-tap next stage pads with ZEROS outside [0, T): intermediate rows at those times are not conv outputs
        auto zero_row_of = [&](int i) {
          if (TAPS2 == 1) return false;
          const int t = (gl * G + i) * S - LEAD + q * 32 + lane;
          return t < 0 || t >= p.Tin || gl > gpi - 1;
        };
        auto taddr_of = [&](int i) { return taddr0 + (uint32_t)(buf * cfg.acc_n[g] + i * Ng); };
        auto dst_of = [&](int i) { return smem + cfg.i_off[g] + bi * cfg.i_bytes[g] + i * cfg.i_tile[g] + (q * 32 + lane) * 16; };
        auto put = [&](int i, int cb, const uint32_t* a, int ncol) {     // <= 16 columns of tile i -> operand rows
          const bool zr = zero_row_of(i);
          uint8_t* const dst = dst_of(i);
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            if (8 * c < ncol) {
              const int chunk = ((col_lo + cb) >> 3) + c;
              uint4 v = epi_chunk8<false>(a + 8 * c, bw + cb + 8 * c, ca, cbk, make_uint4(0u, 0u, 0u, 0u));
              if (zr) v = make_uint4(0u, 0u, 0u, 0u);
              *reinterpret_cast<uint4*>(dst + chunk * (RI * 16)) = v;
            }
          }
        };
        if (GRP && active && wcols == 16) {
          // 16 columns per warp = ONE TMEM load per tile: two tiles of the group are loaded before the wait, or every tile pays
          // a full load latency for ~40 instructions of work
          for (int i = 0; i < G; i += 2) {
            uint32_t a0[16], a1[16];
            tmem_ld16_nowait(taddr_of(i), a0);
            if (i + 1 < G) tmem_ld16_nowait(taddr_of(i + 1), a1);
            tmem_wait_ld();
            put(i, 0, a0, 16);
            if (i + 1 < G) put(i + 1, 0, a1, 16);
          }
        } else if (active) {
          for (int i = 0; i < G; ++i)
            tmem_stream<16>(taddr_of(i), wcols, [&](int cb, const uint32_t (&a)[16], int ncol) { put(i, cb, a, ncol); });
        }
        tc_fence_before();
        fence_async_smem();                                    // generic-proxy writes -> visible to the tensor core's async proxy
        __syncwarp();
        if (lane == 0) {
          mbar_arrive_remote(tempty0_leader + 8u * buf);
          mbar_arrive_remote(ifull0_leader + 8u * bi);
        }
        if (tracer) trace_ev(cp.trace, it, g == 0 ? 5 : 13);
      }
    } else {
      // accumulator of the last GEMM -> the usual fused epilogue to HBM
      constexpr bool POOL = EPI == CE_POOL, RES = EPI == CE_RES;
      PairIter pit(pair0, pair_step, ppi);
      for (int it = 0; it < n_local; ++it, pit.next()) {
        const int gl = group_of(pit.pi);
        const int u = q * 32 + lane;                           // output row of the tile
        const int buf = buf_of(it, nbA);
        if (EPI == CE_HEAD) {
          // Output head: column 0 of the accumulator is the k7 32 -> 1 conv; + bias + the linear x2 interpolation of the
          // low-rate input (App. B.3: x[s] weight 0.75, the neighbour 0.25, edge-clamped), written as plain fp32 [B][Tout].
          // The low-rate samples of all tiles of the group are requested before the accumulator is awaited.
          const int Tout = cp.pl.Tout, Tl = Tout >> 1;
          const bool mine = active && col_lo == 0;
          const int t0 = gl * G * S + u;
          float x0[4], x1[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            x0[i] = x1[i] = 0.f;
            const int t = t0 + i * S;
            if (i < G && mine && u < S && t < Tout) {
              const float* xl = cp.head_xlr + (long long)pit.b * Tl;
              const int s2 = t >> 1;
              const int nb = (t & 1) ? (s2 + 1 < Tl ? s2 + 1 : Tl - 1) : (s2 > 0 ? s2 - 1 : 0);
              x0[i] = __ldg(xl + s2);
              x1[i] = __ldg(xl + nb);
            }
          }
          mbar_wait(tfull_bar(g, buf), phase_of(it, nbA));
          tc_fence_after();
          if (tracer) trace_ev(cp.trace, it, 6);
          const float b0 = s_bias[bias_off];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int t = t0 + i * S;
            if (i < G && mine) {
              uint32_t a[16];
              tmem_ld16_nowait(taddr0 + (uint32_t)(buf * cfg.acc_n[g] + i * Ng), a);
              tmem_wait_ld();
              if (u < S && t < Tout) __stcs(cp.head_y + (long long)pit.b * Tout + t, __uint_as_float(a[0]) + b0 + 0.75f * x0[i] + 0.25f * x1[i]);
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(tempty0_leader + 8u * buf);
          if (tracer) trace_ev(cp.trace, it, 7);
          continue;
        }
        auto row_of = [&](int i) {
          const int t = (gl * G + i) * S + u;                  // >= Tin for a dead tile => every store is masked
          EpiRow row = epi_row<MODE_SAME, POOL, RES>(cp.pl, pit.b, t, col_lo);
          if (TAPS2 > 1) {                                     // rows S .. 127 of a stride-S tile have no output
            row.ok0 = row.ok0 && u < S;
            row.pok = row.pok && u < S;
          }
          return row;
        };
        auto taddr_of = [&](int i) { return taddr0 + (uint32_t)(buf * cfg.acc_n[g] + i * Ng); };
        const float* const bias_w = s_bias + bias_off + col_lo;
        if (GRP && RES) {
          // Residual rows of ALL tiles of the group (the chain's own input: L2 hits, ~700 cycles) are requested before the
          // accumulator is awaited; fetched tile by tile behind the wait they cost a load latency per tile (pipeline trace:
          // 3 900 cycles of epilogue per 4-tile group, the slowest stage of the chain).  Tile i of the group is tile 0 shifted
          // by i * S rows of the same item: one address computation, per tile only the masks.
          const EpiRow base = row_of(0);
          const int t0 = gl * G * S + u;
          uint4 res[4][2];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
#pragma unroll
            for (int c = 0; c < 2; ++c)
              res[i][c] = (i < G && active && t0 + i * S < cp.pl.Tin) ? __ldcs(reinterpret_cast<const uint4*>(base.rrow + (long long)i * S * 8 + c * base.rstride))
                                                                     : make_uint4(0u, 0u, 0u, 0u);
          }
          mbar_wait(tfull_bar(g, buf), phase_of(it, nbA));
          tc_fence_after();
          if (tracer) trace_ev(cp.trace, it, 6);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (i < G && active) {
              EpiRow r = base;
              const int t = t0 + i * S;
              r.in_ok = t < cp.pl.Tin;
              r.ok0 = r.in_ok && t < cp.pl.Tout && u < S;
              r.o0 += (long long)i * S * 16;
              uint32_t a[16];                                  // the residual epilogue has <= 32 columns: 16 per warp, one load
              tmem_ld16_nowait(taddr_of(i), a);
              tmem_wait_ld();
              epi_store_block<MODE_SAME, POOL, RES, 16>(r, bias_w, 0, a, 16, 0.5f * (1.0f + slope), 0.5f * (1.0f - slope), res[i]);
            }
          }
        } else {
          for (int i = 0; i < G; ++i) {
            const EpiRow row = row_of(i);
            uint4 resv[2];
            epi_prefetch_res<RES>(row, active, resv);          // residual rows (the chain's own input: L2 hits) before the wait
            if (i == 0) {
              mbar_wait(tfull_bar(g, buf), phase_of(it, nbA));
              tc_fence_after();
              if (tracer) trace_ev(cp.trace, it, 6);
            }
            if (active) epi_store<MODE_SAME, POOL, RES, 16>(row, bias_w, taddr_of(i), wcols, slope, resv);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(tempty0_leader + 8u * buf);
        if (tracer) trace_ev(cp.trace, it, 7);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 1) tmem_dealloc2(tmem_base, (uint32_t)cfg.tmem_cols);
}

// ----------------------------------------------------------------------------- host side
int chain_tile_stride(int taps2) { return TILE_M - ((taps2 > 1 ? taps2 : 1) - 1); }

// tiles per group for a chain: narrow k3 chains (every GEMM at most 64 columns wide) take as many as TMEM allows, up to 4
static int chain_group_tiles(const ChainParams& cp) {
  if (cp.n_gemms != 2 || (cp.p.taps != 3 && cp.p.taps != 5) || cp.N[0] > 64 || cp.N[1] > 64) return 1;
  int G = 4;
  while (G > 1 && 2 * G * (cp.N[0] + cp.N[1]) > 512) G >>= 1;
  return G;
}

static bool pick_chain_cfg(const ChainParams& cp, ChainCfg& c) {
  const ConvParams& p = cp.p;
  const int NG = cp.n_gemms;
  const int taps2 = cp.taps2 > 1 ? cp.taps2 : 1;
  const int S = chain_tile_stride(taps2);
  for (int G = chain_group_tiles(cp); G >= 1; G >>= 1) {
    c.G = G;
    c.R = (G - 1) * S + TILE_M + (p.taps - 1) * p.dil;
    c.RI = TILE_M + (taps2 - 1);
    int off = 0, cols = 0;
    for (int g = 0; g < NG; ++g) {
      const int K = g == 0 ? p.Cin * p.taps : cp.N[g - 1] * (g == 1 ? taps2 : 1);
      c.w_bytes[g] = K * (cp.N[g] / 2) * 2;
      c.w_off[g] = off;
      off += (c.w_bytes[g] + 1023) / 1024 * 1024;
      // two GEMMs: both accumulators double-buffered; three GEMMs: G1 and G2 rotate through the same two buffers, G3 single
      c.nbA[g] = g == 2 ? 1 : 2;
      c.acc_n[g] = G * cp.N[g];
      if (NG == 3 && g == 1) { c.acc_col[1] = c.acc_col[0]; continue; }
      c.acc_col[g] = cols;
      cols += c.nbA[g] * c.acc_n[g];
    }
    if (cols > 512) continue;
    int tc = 32;
    while (tc < cols) tc <<= 1;
    c.tmem_cols = tc;
    const int w_end = off;
    // Every stage costs the issuer a barrier round trip (~200 cycles) and the tensor pipe's queue is only ~6 MMAs deep, so
    // stages are as large as still leaves >= 4 of them (the L2 prefetch, not the ring, covers HBM latency); the
    // intermediate operand is double-buffered when that still fits.
    for (int kbs = 4; kbs >= 1; kbs >>= 1) {
      if (p.Cin % (16 * kbs)) continue;
      for (int nbi = (NG == 2 ? 2 : 1); nbi >= 1; nbi >>= 1) {
        off = w_end;
        for (int g = 0; g < NG - 1; ++g) {
          c.nbI[g] = nbi;
          c.i_tile[g] = (cp.N[g] / 8) * c.RI * 16;
          c.i_bytes[g] = G * c.i_tile[g];
          c.i_off[g] = off;
          off += c.nbI[g] * c.i_bytes[g];
        }
        c.stage_off = off;
        const int room = CH_SMEM_BUDGET - CH_BAR_BYTES - CH_BIAS_BYTES - off;
        c.kbs = kbs;
        c.stage_bytes = kbs * 2 * c.R * 16;
        int stages = room / c.stage_bytes;
        if (stages > CH_MAX_STAGES) stages = CH_MAX_STAGES;
        if (stages >= 4 || (kbs == 1 && stages >= 2)) {
          c.stages = stages;
          c.nks = p.Cin / (16 * kbs);
          c.bar_off = c.stage_off + stages * c.stage_bytes;
          c.bar_off = (c.bar_off + 15) / 16 * 16;
          c.bias_off = c.bar_off + CH_BAR_BYTES;
          c.smem_bytes = c.bias_off + CH_BIAS_BYTES;
          return true;
        }
      }
    }
  }
  return false;
}

bool conv_chain_fits(int Cin, int taps, int dil, const int* N, int n_gemms, int taps2) {
  if (n_gemms < 2 || n_gemms > 3 || (taps != 3 && taps != 5 && taps != 7)) return false;
  if (taps == 7 && taps2 != 7) return false;                                      // k7 only as the k7 -> k7 decoder pair
  if (taps == 5 && taps2 != 7) return false;                                      // k5 only in front of the k7 output head
  if (taps2 != 1 && ((taps2 != taps && taps != 5) || n_gemms != 2 || dil != 1)) return false;
  if (n_gemms == 3 && N[0] != N[1]) return false;    // G1 and G2 rotate through the same accumulator buffers
  for (int g = 0; g + 1 < n_gemms; ++g)
    if (N[g] > 128) return false;                     // an intermediate operand is at most 128 channels wide
  ChainParams cp{};
  cp.p.Cin = Cin; cp.p.taps = taps; cp.p.dil = dil;
  cp.n_gemms = n_gemms;
  cp.taps2 = taps2;
  for (int g = 0; g < n_gemms; ++g) cp.N[g] = N[g];
  ChainCfg cfg;
  if (!pick_chain_cfg(cp, cfg)) return false;
  // A k3 -> k3 pair whose resident weights leave only a short activation ring runs slower fused than as two launches
  // (measured: the U-Net's 256 -> 128 -> 128 decoder pair, 147 KB of weights per CTA: 5.5 ms vs 3.5 ms per 1184-chunk step)
  if (taps2 > 1 && cfg.w_bytes[0] + cfg.w_bytes[1] > 128 * 1024) return false;
  return true;
}

int launch_conv_chain(const ChainParams& cp, cudaStream_t stream) {
  const ConvParams& p = cp.p;
  const int NG = cp.n_gemms;
  const int taps2 = cp.taps2 > 1 ? cp.taps2 : 1;
  AR_CHECK(NG == 2 || NG == 3, AR_ERR_INVALID, "conv_chain: 2 or 3 GEMMs");
  AR_CHECK(p.Cin % 16 == 0 && p.mode == MODE_SAME && p.pool == nullptr && p.res == nullptr, AR_ERR_INVALID, "conv_chain: unsupported first layer");
  AR_CHECK(p.pad_left <= HALO && (p.taps - 1) * p.dil - p.pad_left <= HALO, AR_ERR_INVALID, "conv_chain: conv reach exceeds HALO");
  AR_CHECK(taps2 == 1 || ((taps2 == p.taps || (p.taps == 5 && taps2 == 7)) && NG == 2 && p.dil == 1 && p.pad_left == (p.taps - 1) / 2),
           AR_ERR_INVALID, "conv_chain: a k-tap second stage is implemented for k3 -> k3, k7 -> k7 and k5 -> k7");
  AR_CHECK(p.pad_left + (taps2 - 1) / 2 <= HALO, AR_ERR_INVALID, "conv_chain: combined reach exceeds HALO");
  int nb = 0;
  for (int g = 0; g < NG; ++g) {
    AR_CHECK(cp.N[g] % 32 == 0 && cp.N[g] >= 32 && cp.N[g] <= 256, AR_ERR_INVALID, "conv_chain: unsupported channel count");
    AR_CHECK(g == NG - 1 || cp.N[g] <= 128, AR_ERR_INVALID, "conv_chain: intermediate wider than 128 channels");
    nb += cp.N[g];
  }
  AR_CHECK(NG == 2 || cp.N[0] == cp.N[1], AR_ERR_INVALID, "conv_chain: the first two GEMMs of a three-GEMM chain share their accumulator buffers");
  AR_CHECK(nb * 4 <= CH_BIAS_BYTES, AR_ERR_INVALID, "conv_chain: too many bias entries");
  const int epi = cp.head_y != nullptr ? CE_HEAD : cp.pl.pool != nullptr ? CE_POOL : (cp.pl.res != nullptr ? CE_RES : CE_PLAIN);
  AR_CHECK(epi != CE_HEAD || (cp.head_xlr != nullptr && cp.pl.pool == nullptr && cp.pl.res == nullptr && p.taps == 5 && taps2 == 7),
           AR_ERR_INVALID, "conv_chain: the output-head epilogue belongs to the k5 -> k7 chain");
  AR_CHECK(!(cp.pl.pool && cp.pl.res), AR_ERR_INVALID, "conv_chain: pool and residual epilogues are exclusive");
  AR_CHECK(epi != CE_RES || cp.N[NG - 1] <= 32, AR_ERR_INVALID, "conv_chain: residual epilogue supports at most 32 columns");
  AR_CHECK(p.tiles_per_item == (p.Tin + chain_tile_stride(taps2) - 1) / chain_tile_stride(taps2), AR_ERR_INVALID,
           "conv_chain: tiles_per_item does not match the tile stride");
  ChainCfg cfg;
  AR_CHECK(pick_chain_cfg(cp, cfg), AR_ERR_INVALID, "conv_chain: no configuration fits shared memory / TMEM");
  AR_CHECK(!cp.pl.out_tblock || (cfg.G == 1 && cp.N[NG - 1] > 32), AR_ERR_INVALID, "conv_chain: time-blocked output only for wide ungrouped chains");
  using Kernel = void (*)(ChainParams, ChainCfg, int);
  struct Entry { int taps, ng, taps2, epi, grp; Kernel k; };
  static const Entry table[] = {
      {3, 2, 1, CE_PLAIN, 0, conv_chain_kernel<3, 2, 1, CE_PLAIN, false>}, {3, 3, 1, CE_PLAIN, 0, conv_chain_kernel<3, 3, 1, CE_PLAIN, false>},
      {3, 2, 3, CE_PLAIN, 0, conv_chain_kernel<3, 2, 3, CE_PLAIN, false>}, {3, 2, 3, CE_POOL, 0, conv_chain_kernel<3, 2, 3, CE_POOL, false>},
      {3, 2, 3, CE_RES, 0, conv_chain_kernel<3, 2, 3, CE_RES, false>},     {7, 2, 7, CE_PLAIN, 0, conv_chain_kernel<7, 2, 7, CE_PLAIN, false>},
      {3, 2, 1, CE_PLAIN, 1, conv_chain_kernel<3, 2, 1, CE_PLAIN, true>},  {3, 2, 3, CE_PLAIN, 1, conv_chain_kernel<3, 2, 3, CE_PLAIN, true>},
      {3, 2, 3, CE_POOL, 1, conv_chain_kernel<3, 2, 3, CE_POOL, true>},    {3, 2, 3, CE_RES, 1, conv_chain_kernel<3, 2, 3, CE_RES, true>},
      {5, 2, 7, CE_HEAD, 1, conv_chain_kernel<5, 2, 7, CE_HEAD, true>},    {5, 2, 7, CE_HEAD, 0, conv_chain_kernel<5, 2, 7, CE_HEAD, false>},
  };
  static DeviceOnce attrs;
  if (attrs.pending()) {
    for (const Entry& e : table) AR_CUDA_OK(cudaFuncSetAttribute(e.k, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM_BUDGET));
    attrs.done();
  }
  Kernel kernel = nullptr;
  for (const Entry& e : table)
    if (e.taps == p.taps && e.ng == NG && e.taps2 == taps2 && e.epi == epi && e.grp == (cfg.G > 1 ? 1 : 0)) kernel = e.k;
  AR_CHECK(kernel != nullptr, AR_ERR_INVALID, "conv_chain: no kernel instantiated for this (taps, stages, epilogue) combination");
  const int gpi = (p.tiles_per_item + cfg.G - 1) / cfg.G;      // tile groups per item; a cluster takes two of them per step
  const int ppi = (gpi + 1) / 2;
  const int num_pairs = p.B * ppi;
  int groups = sm_count() / 2;
  if (groups > num_pairs) groups = num_pairs;
  if (groups < 1) groups = 1;
  kernel<<<groups * 2, ch_threads(NG), cfg.smem_bytes, stream>>>(cp, cfg, num_pairs);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

}  // namespace ar
