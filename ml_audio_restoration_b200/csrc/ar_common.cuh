// Shared definitions for libaudiorestore_sm100: activation layout, conv parameters,
// the fused conv epilogue and error plumbing.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include <string>

#include "../../include/audiorestore.h"

namespace ar {

// ----------------------------------------------------------------------------- errors
void set_error(const std::string& msg);
#define AR_CUDA_OK(expr)                                                                    \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      ar::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                    \
      return AR_ERR_CUDA;                                                                   \
    }                                                                                       \
  } while (0)
#define AR_CHECK(cond, code, msg)                                                           \
  do {                                                                                      \
    if (!(cond)) {                                                                          \
      ar::set_error(msg);                                                                   \
      return (code);                                                                        \
    }                                                                                       \
  } while (0)
#define AR_TRY(expr)                                                                        \
  do {                                                                                      \
    int _r = (expr);                                                                        \
    if (_r != AR_OK) return _r;                                                             \
  } while (0)

// ----------------------------------------------------------------------------- layout
// Internal activations are "H8" channel-blocked half precision:  [B][C/8][Tp][8] fp16, where
//   Tp = HALO + round_up(T, TILE_M) + HALO   rows of 16 bytes,
// row (HALO + t) of chunk c holds channels 8c..8c+7 at time t.  One conv tap of an implicit-GEMM tile is
// then a contiguous run of rows, so a tile is fetched with one bulk (TMA) copy per channel chunk and every
// tap is a 16-byte-granular shift of the UMMA shared-memory descriptor.  fp16 carries the same 11-bit
// significand as TF32 (the tensor core would drop the rest anyway) at half the bytes and twice the K per
// MMA; values are rounded to nearest and clamped to the fp16 range when stored.  Rows outside [0,T) hold
// garbage in HBM; consumers zero them in shared memory (conv zero padding), producers never write them.
constexpr int TILE_M = 128;
constexpr int HALO = 8;  // >= max one-sided conv reach: dilation 8 * (3-1)/2
constexpr float LRELU_SLOPE = 0.2f;
constexpr float HALF_MAX = 65504.0f;

__host__ __device__ inline int round_up(int a, int b) { return (a + b - 1) / b * b; }
__host__ __device__ inline int padded_rows(int T) { return HALO + round_up(T, TILE_M) + HALO; }

struct Act {      // an H8 (fp16) activation tensor
  void* base = nullptr;   // element (b=0, chunk 0, row 0 == t=-HALO)
  int C = 0;              // channels of the whole buffer
  int T = 0;              // valid length
  int Tp = 0;             // padded rows per chunk
  long long bs = 0;       // halves between batch items = C*Tp
  __host__ __device__ __half* h() const { return reinterpret_cast<__half*>(base); }
};

// element (half) offset; `chunk` counts 8-channel groups
__device__ __forceinline__ long long act_off(long long bs, int Tp, int b, int chunk, int t) {
  return (long long)b * bs + ((long long)chunk * Tp + (HALO + t)) * 8;
}

// Time-blocked H8 ("TB8"): [B][Tp/8][C/8][8 steps][8] -- all channels of 8 consecutive time steps are one
// contiguous (C*16)-byte run.  Used for the LSTM gate pre-activations only: the recurrence streams a
// sequence strictly in time order, and 4 KB runs are what HBM likes (plain H8 would be 128-byte pieces).
__device__ __forceinline__ long long act_off_tb(long long bs, int C8, int b, int chunk, int t) {
  const int tr = HALO + t;
  return (long long)b * bs + (((long long)(tr >> 3) * C8 + chunk) * 8 + (tr & 7)) * 8;
}

__device__ __forceinline__ uint32_t pack_half2(float a, float b) {  // round to nearest, saturate to the finite fp16 range: one F2FP
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// two fp32 values in one 64-bit register pair: operands of the packed 2-wide fp32 instructions (add / mul / fma.rn.f32x2)
__device__ __forceinline__ unsigned long long f2_pack(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint4 pack_half8(const float (&v)[8]) {
  return make_uint4(pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]), pack_half2(v[6], v[7]));
}
__device__ __forceinline__ void unpack_half8(uint4 u, float (&v)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(h[i]);
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}

__device__ __forceinline__ float to_tf32(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}

// ----------------------------------------------------------------------------- conv params
enum ConvMode { MODE_SAME = 0, MODE_INTERLEAVE2 = 1 };

struct ConvParams {
  // input (H8)
  const __half* in;
  long long in_bs;
  int in_Tp, in_coff8;   // chunk offset of the first input channel
  int Tin;               // valid input length; GEMM rows are input time positions
  int Cin;               // multiple of 16
  int taps, dil, pad_left;  // tap j reads input row t + j*dil - pad_left
  // weights, packed for the UMMA B operand: [n_slices][Cin/16][taps][2][N/n_slices][8] fp16
  const __half* w;
  const float* bias;     // [N] fp32
  int N;                 // GEMM N, multiple of 16, <= 256
  int n_slices;          // column slices the weights are packed in (each is one CTA's resident operand)
  int cta2;              // packed for the 2-CTA engine: slices (2i, 2i+1) are the two halves of pair-slice i
  // output (H8)
  int mode;              // MODE_SAME: out[t]; MODE_INTERLEAVE2: cols [0,N/2)->out[2t], [N/2,N)->out[2t+1]
  __half* out;
  long long out_bs;
  int out_Tp, out_coff8;
  int out_tblock;        // write the time-blocked variant of H8 (act_off_tb) instead -- LSTM gate pre-activations
  int Tout;              // valid output length
  __half* pool;          // optional max-pool(2,2) copy of the output (MODE_SAME only), H8
  long long pool_bs;
  int pool_Tp, pool_coff8;
  const __half* res;     // optional residual added after the activation (same geometry as out), H8
  long long res_bs;
  int res_Tp, res_coff8;
  int lrelu;             // LeakyReLU(0.2) after bias
  int B;
  int tiles_per_item;    // ceil(Tin / TILE_M)
};
// Fused epilogue for 8 consecutive GEMM columns [n0, n0+8) of GEMM row t (batch item b), shared by the
// CUDA-core cross-check engine.  Must be called by all 32 lanes of a warp whose lanes hold consecutive rows
// (the pool path exchanges neighbours with shuffles); `acc` = raw accumulators, `resv` = residual operand.
__device__ __forceinline__ void epilogue_chunk8(const ConvParams& p, int b, int t, int n0, const float (&acc)[8], const float (&resv)[8]) {
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    v[i] = acc[i] + p.bias[n0 + i];
    if (p.lrelu) v[i] = v[i] > 0.f ? v[i] : LRELU_SLOPE * v[i];
    if (p.res != nullptr) v[i] += resv[i];
  }
  int trow, col;
  if (p.mode == MODE_SAME) {
    trow = t;
    col = n0;
  } else {
    const int half = p.N >> 1;
    const int phase = n0 >= half;
    trow = 2 * t + phase;
    col = n0 - phase * half;
  }
  const bool row_ok = (t < p.Tin) && (trow < p.Tout);
  __half* o = p.out;
  const uint4 packed = pack_half8(v);
  if (row_ok) {
    const long long off = p.out_tblock ? act_off_tb(p.out_bs, p.N >> 3, b, col >> 3, trow)
                                       : act_off(p.out_bs, p.out_Tp, b, p.out_coff8 + (col >> 3), trow);
    *reinterpret_cast<uint4*>(o + off) = packed;
  }
  if (p.mode == MODE_INTERLEAVE2 && t == p.Tin - 1 && 2 * p.Tin < p.Tout && n0 < (p.N >> 1))
    *reinterpret_cast<uint4*>(o + act_off(p.out_bs, p.out_Tp, b, p.out_coff8 + (col >> 3), 2 * p.Tin)) = make_uint4(0u, 0u, 0u, 0u);
  if (p.pool != nullptr) {  // MaxPool1d(2,2), floor; max of the ROUNDED values == rounded max (rounding is monotonic)
    float r[8], m[8];
    unpack_half8(packed, r);
#pragma unroll
    for (int i = 0; i < 8; ++i) m[i] = fmaxf(r[i], __shfl_down_sync(0xffffffffu, r[i], 1));
    if (((t & 1) == 0) && (t + 1 < p.Tin))
      *reinterpret_cast<uint4*>(p.pool + act_off(p.pool_bs, p.pool_Tp, b, p.pool_coff8 + (col >> 3), t >> 1)) = pack_half8(m);
  }
}

// A fused chain (conv_chain.cu): first GEMM = `p` (k-tap conv, input geometry, W1, bias1), then n_gemms-1 further convs
// (pointwise, or one k3 conv: taps2 = 3) whose inputs never leave the SM.  `pl` carries the output geometry of the LAST
// stage (out*, Tout, out_tblock, pool*, res*, N = N[n_gemms-1]); every stage's weights are packed as one 2-CTA pair-slice
// (two column halves).  p.tiles_per_item counts tiles of chain_tile_stride(taps2) rows.
struct ChainParams {
  ConvParams p, pl;
  int n_gemms;
  int taps2;          // taps of the second GEMM: 1 (pointwise), or k (tile stride 128 - (k - 1): k3 -> k3 126, k7 behind it 122)
  float* head_y;      // CE_HEAD chains (k5 -> k7 output head): plain fp32 output [B][Tout], column 0 of the last GEMM ...
  const float* head_xlr;   // ... plus the linear x2 interpolation of this low-rate signal [B][Tout / 2] (super_resolution.py:96-99)
  const __half* w[3];
  const float* bias[3];
  int N[3];
  int lrelu[3];
  long long* trace;   // optional pipeline trace buffer (ar_debug_chain_trace), else nullptr
};

// ----------------------------------------------------------------------------- launchers
bool conv_chain_fits(int Cin, int taps, int dil, const int* N, int n_gemms, int taps2);   // shape / shared memory / TMEM check
int chain_tile_stride(int taps2);                                   // output rows per tile: 128, or 126 behind a k3 second stage
int launch_conv_chain(const ChainParams& cp, cudaStream_t stream);  // fused k-tap conv -> conv(s), 2-CTA engine
int launch_conv_umma2(const ConvParams& p, cudaStream_t stream);   // the tcgen05 engine (cta_group::2; needs p.cta2)
int launch_conv_simt(const ConvParams& p, cudaStream_t stream);    // CUDA-core cross-check engine

// ----------------------------------------------------------------------------- per-device host state (device.cu)
int current_device();
int sm_count();            // of the CURRENT device
// "Done once" flag kept per device: kernel attributes (opt-in dynamic shared memory, carve-out) are per device / context,
// so a process that drives cuda:0 and cuda:1 must set them on both.
//   static DeviceOnce once;  if (once.pending()) { cudaFuncSetAttribute(...); once.done(); }
struct DeviceOnce {
  static constexpr int MAX_DEVICES = 64;
  std::atomic<unsigned long long> bits{0};
  bool pending() const;
  void done();
};

}  // namespace ar
