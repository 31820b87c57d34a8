// 2-CTA (cta_group::2) variant of the tcgen05 implicit-GEMM Conv1d engine.
//
// A cluster of two CTAs (an SM pair) computes TWO adjacent 128-row time tiles with ONE instruction
// stream: D[256 x Ns] (fp32, TMEM) += A[256 x 16] * B[16 x Ns] (fp16) per `tcgen05.mma.cta_group::2.kind::f16`.  Each CTA keeps in its
// own shared memory (a) the activation rows of its own tile (same H8 / no-swizzle K-major layout and
// tap-shift trick as conv_umma.cu) and (b) HALF of the weight columns (Ns/2), and in its own TMEM the
// 128 accumulator rows of its tile.  Compared with the 1-CTA kernel this halves the number of MMA
// instructions per tile (the layers here are bound by the fixed per-MMA operand fetch, not by FLOPs)
// and halves the resident weight bytes per CTA, so 128->128 k3, 128->64 k7 ... layers need no N-slices.
//
// Roles per CTA: warp 0 = bulk-copy (TMA) producer for its own rows, warp 1 = "MMA warp", warps 2..9 =
// epilogue for its own 128 rows.  Only the leader CTA's (rank 0) MMA warp issues tcgen05.mma; the
// peer's MMA warp zero-pads its edge rows and then tells the leader, per pipeline stage, that its half
// of the operands is in place (remote mbarrier arrive).  Stage release (empty) and accumulator-ready
// (tmem_full) are multicast commits that arrive in both CTAs; accumulator-drained (tmem_empty) is
// collected in the leader from the epilogue warps of both CTAs.
#include "ar_common.cuh"
#include "umma_ptx.cuh"
#include "umma_epilogue.cuh"

namespace ar {

constexpr int EPI2_WARPS = 8;
constexpr int UMMA2_THREADS = 64 + 32 * EPI2_WARPS;
constexpr int SMEM2_BUDGET = 227 * 1024;
constexpr int BAR2_BYTES = 512;
constexpr int BIAS2_BYTES = 1024;
constexpr int UMMA2_PREFETCH = 2;   // tile pairs the L2 prefetch runs ahead of the shared-memory ring

struct Umma2Cfg {
  int kbs, stages, R;
  int w_bytes;      // resident weights per CTA: Cin*taps*(Ns/2)*2
  int stage_bytes;  // activation stage per CTA
  int ncol, tmem_cols, nks, smem_bytes;
  int nbuf;         // TMEM accumulator buffers (2..8): how many tile groups the MMAs may run ahead of the epilogue
  int G;            // tiles per CTA per group (1, 2 or 4): each CTA owns G consecutive 128-row tiles of a group, loaded as ONE
                    // run of rows per channel chunk; the barrier round trips of a stage / an accumulator are paid once per
                    // group, which is what bounds the layers with few MMAs per tile (Cin <= 64, k <= 3)
  int RG;           // rows of a group's run: G*128 + (taps-1)*dil
  int res_off, res_bytes;   // residual epilogue: two-deep shared-memory ring of the group's residual rows (bulk-copied by the producer)
};

// Rows of CTA `rank`'s run for group `gi` of an item: first row (time index, may be negative), how many rows exist in the
// buffer from there (the run is clamped to the padded chunk), and whether every tile of the run lies beyond the item
// (then a valid run is loaded instead and all rows are zeroed).
struct RunGeom { int t_start, rows, tile0; bool all_dead; };
__device__ __forceinline__ RunGeom run_geom(const ConvParams& p, const Umma2Cfg& cfg, int gi, int rank) {
  RunGeom g;
  g.tile0 = (gi * 2 + rank) * cfg.G;
  g.all_dead = g.tile0 > p.tiles_per_item - 1;
  const int tl = g.all_dead ? p.tiles_per_item - 1 : g.tile0;
  g.t_start = tl * TILE_M - p.pad_left;
  const int avail = p.in_Tp - (HALO + g.t_start);
  g.rows = cfg.RG < avail ? cfg.RG : avail;
  return g;
}

template <int MODE, bool POOL, bool RES, int TAPS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(UMMA2_THREADS, 1)
conv_umma2_kernel(const __grid_constant__ ConvParams p, const __grid_constant__ Umma2Cfg cfg, int num_pairs) {
  extern __shared__ __align__(1024) uint8_t smem[];
  // shared memory (identical offsets in both CTAs): [weight half][stages x activation stage][barriers][bias]
  const uint32_t w_base = smem_u32(smem);
  const uint32_t smem_base = w_base + cfg.w_bytes;
  uint8_t* const stage_ptr = smem + cfg.w_bytes;
  const uint32_t bar_base = smem_base + cfg.stages * cfg.stage_bytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (cfg.stages + s); };
  auto rfull_bar = [&](int i) { return bar_base + 8u * (2 * cfg.stages + i); };        // residual ring (RES kernels)
  auto rempty_bar = [&](int i) { return bar_base + 8u * (2 * cfg.stages + 2 + i); };
  auto tfull_bar = [&](int i) { return bar_base + 8u * (3 * cfg.stages + i); };
  auto tempty_bar = [&](int i) { return bar_base + 8u * (3 * cfg.stages + 8 + i); };  // used in the leader only
  const uint32_t w_bar = bar_base + 8u * (3 * cfg.stages + 16);
  volatile uint32_t* tmem_slot =
      reinterpret_cast<volatile uint32_t*>(stage_ptr + cfg.stages * cfg.stage_bytes + 8 * (3 * cfg.stages + 17));
  float* const s_bias = reinterpret_cast<float*>(stage_ptr + cfg.stages * cfg.stage_bytes + BAR2_BYTES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < cfg.stages; ++s) {
      // the leader's "stage full" also collects the peer's "my rows have landed" arrive: ONE barrier round trip per
      // stage for the issuing thread (a pipeline trace showed ~200 cycles per wait, more than the stage's MMAs cost to issue)
      mbar_init(full_bar(s), leader ? 2 : 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int i = 0; i < cfg.nbuf; ++i) {
      mbar_init(tfull_bar(i), 1);
      mbar_init(tempty_bar(i), 2 * EPI2_WARPS);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(rfull_bar(i), 1);
      mbar_init(rempty_bar(i), EPI2_WARPS);
    }
    mbar_init(w_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc2(smem_u32((const void*)tmem_slot), (uint32_t)cfg.tmem_cols);
  const int nsl = p.n_slices >> 1;                       // pair-slices (p.n_slices counts per-CTA halves)
  const int Ns = p.N / nsl;                              // GEMM columns of this pair's weight slice
  const int Nh = Ns >> 1;                                // weight columns resident in this CTA
  const int cid = blockIdx.x >> 1;                       // cluster index
  const int slice = cid % nsl;
  for (int i = threadIdx.x; i < Ns; i += blockDim.x) s_bias[i] = p.bias[slice * Ns + i];
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                    // barriers of both CTAs initialised before any remote use
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int tpi = p.tiles_per_item;
  const int ppi = (tpi + 2 * cfg.G - 1) / (2 * cfg.G);   // tile groups (2G tiles: G per CTA) per batch item
  const int RG = cfg.RG;
  const int pair0 = cid / nsl;
  const int pair_step = (gridDim.x >> 1) / nsl;
  const int n_local = pair0 < num_pairs ? (num_pairs - pair0 + pair_step - 1) / pair_step : 0;

  if (warp == 0) {
    // ------------------------------------------------------------------ producer (own rows, own weight half)
    if (elect_one()) {
      mbar_expect_tx(w_bar, (uint32_t)cfg.w_bytes);
      const char* wsrc = reinterpret_cast<const char*>(p.w) + ((size_t)slice * 2 + rank) * cfg.w_bytes;
      for (int off = 0; off < cfg.w_bytes; off += 32768) {
        const int n = cfg.w_bytes - off < 32768 ? cfg.w_bytes - off : 32768;
        bulk_g2s(w_base + off, wsrc + off, (uint32_t)n, w_bar);
      }
      int s = 0;
      uint32_t ph = 0;
      const long long chunk_stride = (long long)p.in_Tp * 8;             // halves between 8-channel chunks
      const int chunks_per_stage = cfg.kbs * 2;
      PairIter pit(pair0, pair_step, ppi), pre(pair0, pair_step, ppi);
      // HBM -> L2 prefetch runs UMMA2_PREFETCH groups ahead of the shared-memory ring (which then only has to cover L2 latency)
      const int n_chunks = p.Cin >> 3;
      const int pre_dist = cfg.G >= 2 ? 2 : UMMA2_PREFETCH;
      for (int d = 0; d < pre_dist && d < n_local; ++d, pre.next()) {
        const RunGeom g = run_geom(p, cfg, pre.pi, (int)rank);
        const __half* ps = p.in + act_off(p.in_bs, p.in_Tp, pre.b, p.in_coff8, g.t_start);
        for (int c = 0; c < n_chunks; ++c, ps += chunk_stride) bulk_prefetch_l2(ps, (uint32_t)(g.rows * 16));
      }
      for (int it = 0; it < n_local; ++it, pit.next()) {
        const RunGeom g = run_geom(p, cfg, pit.pi, (int)rank);
        const __half* src = p.in + act_off(p.in_bs, p.in_Tp, pit.b, p.in_coff8, g.t_start);
        const uint32_t row_bytes = (uint32_t)(g.rows * 16);
        const bool do_pre = it + pre_dist < n_local;
        const __half* ps = nullptr;
        uint32_t pre_bytes = 0;
        if (do_pre) {
          const RunGeom gp = run_geom(p, cfg, pre.pi, (int)rank);
          ps = p.in + act_off(p.in_bs, p.in_Tp, pre.b, p.in_coff8, gp.t_start);
          pre_bytes = (uint32_t)(gp.rows * 16);
          pre.next();
        }
        for (int ks = 0; ks < cfg.nks; ++ks) {
          const uint32_t fb = full_bar(s);
          mbar_wait(empty_bar(s), ph ^ 1u);
          mbar_expect_tx(fb, (uint32_t)chunks_per_stage * row_bytes);
          uint32_t dst = smem_base + s * cfg.stage_bytes;
          for (int c = 0; c < chunks_per_stage; ++c) {
            bulk_g2s(dst, src, row_bytes, fb);
            if (do_pre) { bulk_prefetch_l2(ps, pre_bytes); ps += chunk_stride; }
            dst += (uint32_t)(RG * 16);
            src += chunk_stride;
          }
          if (++s == cfg.stages) { s = 0; ph ^= 1u; }
        }
        if (RES) {
          // The residual operand of the group's epilogue: rows [tile0*128, +G*128) of Ns/8 chunks, bulk-copied into a
          // two-deep ring (a per-thread global load in the epilogue keeps only ~8 KB in flight per SM, far too little
          // to cover the memory latency -- measured 2.5x the time of the same layer without residual).
          const int rb = it & 1;
          const uint32_t rph = (uint32_t)(it >> 1) & 1u;
          mbar_wait(rempty_bar(rb), rph ^ 1u);
          const int t_res = g.tile0 * TILE_M;
          int rows_res = p.res_Tp - (HALO + t_res);
          if (rows_res > cfg.G * TILE_M) rows_res = cfg.G * TILE_M;
          if (g.all_dead || rows_res <= 0) {
            mbar_arrive(rfull_bar(rb));                              // nothing to fetch: every store of the group is masked
          } else {
            const int nch = Ns >> 3;
            mbar_expect_tx(rfull_bar(rb), (uint32_t)(nch * rows_res * 16));
            const __half* pr = p.res + act_off(p.res_bs, p.res_Tp, pit.b, p.res_coff8 + ((slice * Ns) >> 3), t_res);
            uint32_t dst = w_base + cfg.res_off + rb * cfg.res_bytes;
            for (int c = 0; c < nch; ++c) {
              bulk_g2s(dst, pr, (uint32_t)(rows_res * 16), rfull_bar(rb));
              dst += (uint32_t)(cfg.G * TILE_M * 16);
              pr += (long long)p.res_Tp * 8;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA warp
    const uint32_t idesc = make_idesc_f16(256, Ns);          // M = 256: both CTAs' 128 rows
    const uint64_t a_desc_hi = make_desc(0u, (uint32_t)(RG * 16), 128u);
    const uint64_t b_desc_hi = make_desc(0u, (uint32_t)(Nh * 16), 128u);
    mbar_wait(w_bar, 0);
    int s = 0, buf = 0;
    uint32_t ph = 0, aph = 0;
    const uint32_t b_step = (uint32_t)(Nh * 2);
    const uint32_t a_step = (uint32_t)(2 * RG);
    const uint32_t w_addr0 = w_base >> 4;
    const uint32_t dil_u = (uint32_t)p.dil;
    const uint32_t full0_leader = mapa_u32(full_bar(0), 0);
    const int G = cfg.G;
    PairIter pit(pair0, pair_step, ppi);
    for (int it = 0; it < n_local; ++it, pit.next()) {
      const RunGeom g = run_geom(p, cfg, pit.pi, (int)rank);
      const int tfirst = g.t_start;
      const bool dead = g.all_dead;                                    // no such tiles: contribute zeros
      const bool edge = dead || (tfirst < 0) || (tfirst + RG > p.Tin);
      if (leader) {
        mbar_wait(tempty_bar(buf), aph ^ 1u);                          // both epilogues drained this accumulator
        tc_fence_after();
      }
      const uint32_t d_tmem = tmem_base + (uint32_t)(buf * G * cfg.ncol);
      uint32_t b_addr = w_addr0;
      uint32_t accum = 0u;
      for (int ks = 0; ks < cfg.nks; ++ks) {
        mbar_wait(full_bar(s), ph);
        if (edge) {  // conv zero padding of this CTA's rows (and the rows of the run that were never loaded)
          uint8_t* a_ptr = stage_ptr + s * cfg.stage_bytes;
          for (int r = lane; r < RG; r += 32) {
            const int t = tfirst + r;
            if (dead || t < 0 || t >= p.Tin)
              for (int c = 0; c < cfg.kbs * 2; ++c)
                *reinterpret_cast<float4*>(a_ptr + (c * RG + r) * 16) = make_float4(0.f, 0.f, 0.f, 0.f);
          }
          fence_async_smem();
          __syncwarp();
        }
        if (!leader) {
          // my half of this stage (rows + resident weights) is in place: tell the leader
          if (elect_one()) {
            if (edge) mbar_arrive_remote_release(full0_leader + 8u * s);   // zero-padding writes must be visible
            else mbar_arrive_remote(full0_leader + 8u * s);
          }
          __syncwarp();
        } else {
          tc_fence_after();
          if (elect_one()) {
            uint32_t a_addr = (smem_base + s * cfg.stage_bytes) >> 4;
            for (int kb = 0; kb < cfg.kbs; ++kb) {
              for (int gg = 0; gg < G; ++gg) {
                const uint32_t a_g = a_addr + (uint32_t)(gg * TILE_M);          // one tile (128 rows x 16 B) further down the run
                const uint32_t d_g = d_tmem + (uint32_t)(gg * cfg.ncol);
#pragma unroll
                for (int j = 0; j < TAPS; ++j)
                  umma2_f16(d_g, a_desc_hi | (uint64_t)(a_g + (uint32_t)j * dil_u),
                            b_desc_hi | (uint64_t)(b_addr + (uint32_t)j * b_step), idesc, (j == 0) ? accum : 1u);
              }
              accum = 1u;
              b_addr += (uint32_t)TAPS * b_step;
              a_addr += a_step;
            }
            umma_commit2(empty_bar(s));                          // both CTAs' stage s is free once these MMAs retire
            if (ks == cfg.nks - 1) umma_commit2(tfull_bar(buf));   // both accumulator halves ready
          }
          __syncwarp();
        }
        if (++s == cfg.stages) { s = 0; ph ^= 1u; }
      }
      if (++buf == cfg.nbuf) { buf = 0; aph ^= 1u; }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..9), own G x 128 rows
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int wcols = Ns >= 32 ? Ns / 2 : Ns;
    const int col_lo = Ns >= 32 ? half * wcols : 0;
    const bool active = Ns >= 32 || half == 0;
    const float slope = p.lrelu ? LRELU_SLOPE : 1.0f;
    const int gcol0 = slice * Ns + col_lo;
    const uint32_t tempty_leader0 = mapa_u32(tempty_bar(0), 0);   // barriers are 8 bytes apart in the leader too
    const int G = cfg.G;
    int buf = 0;
    uint32_t aph = 0;
    PairIter pit(pair0, pair_step, ppi);
    for (int it = 0; it < n_local; ++it, pit.next()) {
      const int tile0 = (pit.pi * 2 + (int)rank) * G;
      mbar_wait(tfull_bar(buf), aph);
      tc_fence_after();
      const uint4* res_s = nullptr;
      if (RES) {   // this group's residual rows, staged by the producer: [chunk][G*128 rows] x 16 B
        mbar_wait(rfull_bar(it & 1), (uint32_t)(it >> 1) & 1u);
        res_s = reinterpret_cast<const uint4*>(smem + cfg.res_off + (it & 1) * cfg.res_bytes) + (col_lo >> 3) * (G * TILE_M) + q * 32 + lane;
      }
      for (int gg = 0; gg < G; ++gg) {
        const int t = (tile0 + gg) * TILE_M + q * 32 + lane;   // >= Tin for a dead tile => every store is masked
        const EpiRow row = epi_row<MODE, POOL, RES>(p, pit.b, t, gcol0);
        uint4 resv[2];
        if (RES) {
          resv[0] = res_s[gg * TILE_M];
          resv[1] = res_s[G * TILE_M + gg * TILE_M];
        }
        if (active) {
          const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((buf * G + gg) * cfg.ncol + col_lo);
          epi_store<MODE, POOL, RES>(row, s_bias + col_lo, taddr, wcols, slope, resv);
        }
      }
      if (RES) {
        __syncwarp();
        if (lane == 0) mbar_arrive(rempty_bar(it & 1));
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(tempty_leader0 + 8u * buf);   // leader collects 2 x 8 warps
      if (++buf == cfg.nbuf) { buf = 0; aph ^= 1u; }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // no CTA leaves (or frees TMEM) while its peer may still touch it
  if (warp == 1) tmem_dealloc2(tmem_base, (uint32_t)cfg.tmem_cols);
}

// ----------------------------------------------------------------------------- host side
static bool pick_cfg2(const ConvParams& p, Umma2Cfg& c) {
  const int Ns = p.N / (p.n_slices / 2);
  c.R = TILE_M + (p.taps - 1) * p.dil;
  int ncol = 32;
  while (ncol < Ns) ncol <<= 1;
  c.ncol = ncol;
  c.w_bytes = p.Cin * p.taps * (Ns / 2) * 2;
  const int room0 = SMEM2_BUDGET - BAR2_BYTES - BIAS2_BYTES - c.w_bytes;
  for (int kbs = 4; kbs >= 1; kbs >>= 1) {
    if (p.Cin % (16 * kbs)) continue;
    // group size: enough tiles per barrier round that a stage carries >= ~64 MMAs, within TMEM (two buffers) and the ring
    int G = 1;
    // Below 64 MMAs per stage tiles are grouped: also the k7 decoders (28 MMAs per stage) take G = 2 (128 -> 64) / G = 4
    // (64 -> 32) -- fewer barrier round trips per tile and 4-8 KB instead of 2 KB runs per bulk copy (10.8 -> 10.2 ms and
    // 5.3 -> 4.3 ms per launch at 1184 chunks)
    constexpr int kGroupMmas = 64, kMaxGroup = 4;
    while (G < kMaxGroup && kbs * p.taps * G < kGroupMmas && 2 * (2 * G) * ncol <= 512) G *= 2;
    for (; G >= 1; G >>= 1) {
      c.RG = G * TILE_M + (p.taps - 1) * p.dil;
      c.stage_bytes = kbs * 2 * c.RG * 16;
      c.res_bytes = p.res != nullptr ? G * TILE_M * (Ns / 8) * 16 : 0;
      const int room = room0 - 2 * c.res_bytes;
      int stages = room / c.stage_bytes;
      if (stages > 8) stages = 8;
      if (stages >= 4 || (kbs == 1 && G == 1 && stages >= 2)) {
        c.kbs = kbs;
        c.G = G;
        c.stages = stages;
        c.nks = p.Cin / (16 * kbs);
        c.nbuf = 512 / (G * ncol) > 8 ? 8 : 512 / (G * ncol);
        c.tmem_cols = c.nbuf * G * ncol;
        c.res_off = c.w_bytes + stages * c.stage_bytes + BAR2_BYTES + BIAS2_BYTES;
        c.smem_bytes = c.res_off + 2 * c.res_bytes;
        return true;
      }
    }
  }
  return false;
}

int launch_conv_umma2(const ConvParams& p, cudaStream_t stream) {
  AR_CHECK(p.cta2 && p.n_slices >= 2 && (p.n_slices & 1) == 0, AR_ERR_INVALID, "conv_umma2: layer is not packed for the 2-CTA engine");
  const int nsl = p.n_slices / 2;
  const int Ns = p.N / nsl;
  AR_CHECK(p.Cin % 16 == 0 && p.N % (32 * nsl) == 0 && Ns >= 32 && Ns <= 256, AR_ERR_INVALID, "conv_umma2: unsupported channel counts");
  AR_CHECK(p.res == nullptr || Ns <= 32, AR_ERR_INVALID, "conv_umma2: residual epilogue supports at most 32 columns per slice");
  AR_CHECK(p.pad_left <= HALO && (p.taps - 1) * p.dil - p.pad_left <= HALO, AR_ERR_INVALID, "conv_umma2: conv reach exceeds HALO");
  AR_CHECK(p.mode == MODE_SAME || (p.pool == nullptr && p.res == nullptr), AR_ERR_INVALID, "conv_umma2: interleave mode has no pool/residual epilogue");
  AR_CHECK(p.mode == MODE_SAME || (p.N / 2) % (Ns / 2) == 0, AR_ERR_INVALID, "conv_umma2: interleave phases must align with the epilogue column split");
  AR_CHECK(!(p.pool && p.res), AR_ERR_INVALID, "conv_umma2: pool and residual epilogues are exclusive");
  Umma2Cfg cfg;
  AR_CHECK(pick_cfg2(p, cfg), AR_ERR_INVALID, "conv_umma2: no pipeline configuration fits shared memory");
  using Kernel = void (*)(ConvParams, Umma2Cfg, int);
  struct Entry { int variant, taps; Kernel k; };
  static const Entry table[] = {
      {EV_PLAIN, 1, conv_umma2_kernel<MODE_SAME, false, false, 1>}, {EV_PLAIN, 3, conv_umma2_kernel<MODE_SAME, false, false, 3>},
      {EV_PLAIN, 5, conv_umma2_kernel<MODE_SAME, false, false, 5>}, {EV_PLAIN, 7, conv_umma2_kernel<MODE_SAME, false, false, 7>},
      {EV_POOL, 3, conv_umma2_kernel<MODE_SAME, true, false, 3>},   {EV_RES, 3, conv_umma2_kernel<MODE_SAME, false, true, 3>},
      {EV_INTERLEAVE, 1, conv_umma2_kernel<MODE_INTERLEAVE2, false, false, 1>},
      {EV_INTERLEAVE, 3, conv_umma2_kernel<MODE_INTERLEAVE2, false, false, 3>},
  };
  static DeviceOnce attrs;   // per device: function attributes belong to the device's context
  if (attrs.pending()) {
    for (const Entry& e : table) AR_CUDA_OK(cudaFuncSetAttribute(e.k, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM2_BUDGET));
    attrs.done();
  }
  const int variant = epi_variant(p);
  Kernel kernel = nullptr;
  for (const Entry& e : table)
    if (e.variant == variant && e.taps == p.taps) kernel = e.k;
  AR_CHECK(kernel != nullptr, AR_ERR_INVALID, "conv_umma2: no kernel instantiated for this (epilogue, taps) combination");
  const int ppi = (p.tiles_per_item + 2 * cfg.G - 1) / (2 * cfg.G);   // tile groups per item
  const int num_pairs = p.B * ppi;
  int groups = (sm_count() / 2) / nsl;                   // clusters per pair-slice
  if (groups > num_pairs) groups = num_pairs;
  if (groups < 1) groups = 1;
  const int grid = groups * nsl * 2;
  kernel<<<grid, UMMA2_THREADS, cfg.smem_bytes, stream>>>(p, cfg, num_pairs);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

}  // namespace ar
