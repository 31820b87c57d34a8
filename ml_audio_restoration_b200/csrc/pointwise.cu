// CUDA-core kernels around the tensor-core convs: Cin=1 stems, Cout=1 tails (with the fused
// denoiser mask logic and the super-res linear-interp residual), normalize, chunk split and
// overlap-add.  All are HBM-bound streaming passes with coalesced (float4 where the layout
// allows) accesses.
#include <cstring>
#include <vector>

#include "ar_common.cuh"
#include "pointwise.cuh"

namespace ar {

// ============================================================================ stem: Cin = 1
// x[B][T] plain fp32 -> H8 fp16 out (32 channels): conv(k taps, pad k/2) + folded BN bias + LeakyReLU.
// denoiser.py:54 (encoder.0.0), super_resolution.py:25 (initial.0), stereo_separator.py:25.
// Two output channels per instruction: `fma.rn.f32x2` (SASS FFMA2) takes the weight pair (2i, 2i+1) of a tap as ONE 8-byte
// constant-bank / uniform-register operand and broadcasts the input sample, so a k7 stem is 112 FFMA2 instead of 224 FFMA per
// sample (the kernel was FFMA-issue-bound: 470 instructions per sample behind 68 bytes).  Same accumulation order per channel
// as the scalar form (bias, then taps 0..k-1): bit-identical results.
template <int TAPS>
__global__ void __launch_bounds__(128) stem_kernel(const float* __restrict__ x, int T, const __grid_constant__ StemP w,
                                                   __half* __restrict__ out, long long out_bs, int out_Tp, int lrelu) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const float* xb = x + (long long)b * T;
  unsigned long long xin[TAPS];
#pragma unroll
  for (int j = 0; j < TAPS; ++j) {
    const int ti = t + j - TAPS / 2;
    const float v = (ti >= 0 && ti < T) ? __ldg(xb + ti) : 0.f;
    xin[j] = f2_pack(v, v);
  }
  const float slope = lrelu ? LRELU_SLOPE : 1.0f;
  const unsigned long long slope2 = f2_pack(slope, slope);
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      unsigned long long a = f2_pack(w.b[8 * c + 2 * i], w.b[8 * c + 2 * i + 1]), s;
#pragma unroll
      for (int j = 0; j < TAPS; ++j) {
        const unsigned long long wj = f2_pack(w.w[j][8 * c + 2 * i], w.w[j][8 * c + 2 * i + 1]);
        asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a) : "l"(wj), "l"(xin[j]));
      }
      asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(s) : "l"(a), "l"(slope2));
      float a0, a1, s0, s1;
      f2_unpack(a, a0, a1);
      f2_unpack(s, s0, s1);
      v[2 * i] = fmaxf(a0, s0);
      v[2 * i + 1] = fmaxf(a1, s1);
    }
    *reinterpret_cast<uint4*>(out + act_off(out_bs, out_Tp, b, c, t)) = pack_half8(v);
  }
}

int launch_stem(const float* x, int B, int T, const StemP& w, const Act& out, int lrelu, cudaStream_t stream) {
  dim3 grid((T + 127) / 128, B);
  if (w.taps == 3)
    stem_kernel<3><<<grid, 128, 0, stream>>>(x, T, w, out.h(), out.bs, out.Tp, lrelu);
  else if (w.taps == 7)
    stem_kernel<7><<<grid, 128, 0, stream>>>(x, T, w, out.h(), out.bs, out.Tp, lrelu);
  else {
    set_error("stem: unsupported tap count");
    return AR_ERR_INVALID;
  }
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

// ============================================================================ final k7, C(32) -> 1
// y[b][och][t] = bias + sum_{c<32, j<7} w[c][j] * in[c][t+j-3]   (+ linear x2 interpolation of x_lr)
// super_resolution.py:62,96-99 (reconstruction + F.interpolate residual, App. B.3);
// stereo_separator.py:81 ({left,right}_decoder.9) with blockIdx.z selecting the side.
// A block stages 256+6 rows of raw fp16 in shared memory once; every thread produces TWO neighbouring outputs from
// the 8 rows it reads (each row is used by 7 taps x 2 outputs), all 448 FFMAs take their weight as a constant-bank
// operand.  Rows are stored at index r + (r >> 3) so that the 32-byte lane stride of the reads is conflict-free.
struct FinalArgs {
  const __half* in;
  long long in_bs;
  int in_Tp;
  int in_coff8[2];
  float* y;              // [B][nout][T]
  int nout;
  int T;
  const float* x_lr;     // optional [B][T/2] low-rate input for the interp residual
};
constexpr int FK_THREADS = 128;
constexpr int FK_OUT = 2 * FK_THREADS;               // outputs per block
constexpr int FK_ROWS = FK_OUT + 6;
constexpr int FK_PITCH = FK_ROWS + (FK_ROWS >> 3) + 1;

template <int O>
__device__ __forceinline__ void final_k7_rows(const uint4 (*tile)[FK_PITCH], const FinalW& w, int r0, float& acc0, float& acc1) {
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float x[8][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int r = r0 + k;
      unpack_half8(tile[c][r + (r >> 3)], x[k]);
    }
#pragma unroll
    for (int j = 0; j < 7; ++j)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        acc0 = fmaf(x[j][i], w.w[O][j][8 * c + i], acc0);
        acc1 = fmaf(x[j + 1][i], w.w[O][j][8 * c + i], acc1);
      }
  }
}

__global__ void __launch_bounds__(FK_THREADS) final_k7_kernel(const __grid_constant__ FinalArgs a, const __grid_constant__ FinalW w) {
  __shared__ uint4 tile[4][FK_PITCH];
  const int o = blockIdx.z, b = blockIdx.y;
  const int t0 = blockIdx.x * FK_OUT;
  for (int i = threadIdx.x; i < 4 * FK_ROWS; i += FK_THREADS) {
    const int c = i / FK_ROWS, r = i - c * FK_ROWS;
    const int t = t0 - 3 + r;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);                 // conv zero padding
    if (t >= 0 && t < a.T) v = *reinterpret_cast<const uint4*>(a.in + act_off(a.in_bs, a.in_Tp, b, a.in_coff8[o] + c, t));
    tile[c][r + (r >> 3)] = v;
  }
  __syncthreads();
  const int t = t0 + 2 * threadIdx.x;
  if (t >= a.T) return;
  float acc0 = w.bias[o], acc1 = acc0;
  if (o == 0) final_k7_rows<0>(tile, w, 2 * threadIdx.x, acc0, acc1);
  else final_k7_rows<1>(tile, w, 2 * threadIdx.x, acc0, acc1);
  if (a.x_lr != nullptr) {   // F.interpolate(scale 2, linear, align_corners=False): t is even
    const int Tl = a.T >> 1;
    const float* xl = a.x_lr + (long long)b * Tl;
    const int s = t >> 1;
    const float x0 = __ldg(xl + s);
    const float xm = __ldg(xl + (s > 0 ? s - 1 : 0));
    const float x1 = __ldg(xl + (s + 1 < Tl ? s + 1 : Tl - 1));
    acc0 += 0.25f * xm + 0.75f * x0;
    acc1 += 0.75f * x0 + 0.25f * x1;
  }
  float* yo = a.y + ((long long)b * a.nout + o) * a.T + t;
  if (t + 1 < a.T && (reinterpret_cast<uintptr_t>(yo) & 7) == 0) {
    *reinterpret_cast<float2*>(yo) = make_float2(acc0, acc1);
  } else {
    yo[0] = acc0;
    if (t + 1 < a.T) yo[1] = acc1;
  }
}

int launch_final_k7(const Act& in, const int* in_coff8, const FinalW& w, int nout, float* y, int B, int T, const float* x_lr,
                    cudaStream_t stream) {
  FinalArgs a;
  a.in = in.h(); a.in_bs = in.bs; a.in_Tp = in.Tp;
  a.in_coff8[0] = in_coff8[0];
  a.in_coff8[1] = nout > 1 ? in_coff8[1] : in_coff8[0];
  a.y = y; a.nout = nout; a.T = T; a.x_lr = x_lr;
  dim3 grid((T + FK_OUT - 1) / FK_OUT, B, nout);
  final_k7_kernel<<<grid, FK_THREADS, 0, stream>>>(a, w);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

// ============================================================================ denoiser tail
// f (H8, 32 ch) and the raw input x -> y:
//   m_t = sigmoid(conv3(lrelu(conv3(lrelu(conv3(f, 32->16)), 16->8)), 8->1))   denoiser.py:39-46
//   m_i = clamp(box5((2|d2x| + |dx| + .5|x|)/3.5), 0, 1)                        denoiser.py:62-86
//   y   = conv1(f, 32->1) * (1 - 0.9*max(m_t, m_i))                              denoiser.py:134-142
// Every conv zero-pads ITS OWN input at the sequence ends, so intermediate activations are
// forced to zero outside [0,T).  Activations are staged in shared memory (fp32); all weights are constant-bank
// FFMA operands (DenTailP is a kernel parameter).
// PRE = true (product path): the first detector layer (32 -> 16, 1536 of the 1976 MACs per sample) has already run on
// the tensor core as an ordinary conv-engine layer ("td0", padded to 32 columns) and arrives as `h1` (H8, channels
// 0..15); this kernel then costs 440 FFMA per sample instead of 1976 (it was FMA-issue bound: 5.9 ms per 1184-chunk step).
// PRE = false: everything on CUDA cores from f (cross-check engine, AR_DEN_TAIL_SIMT=1).
constexpr int DT = 128;       // threads per block = rows of the first detector layer a block computes
constexpr int DT_OUT = DT - 4;  // outputs per block: 128 td0 rows -> 126 td1 rows -> 124 outputs, one pass per thread each

template <bool PRE>
__global__ void __launch_bounds__(DT) den_tail_kernel(const __half* __restrict__ fin, long long f_bs, int f_Tp,
                                                      const __half* __restrict__ h1, long long h_bs, int h_Tp,
                                                      const float* __restrict__ x, float* __restrict__ y, int T,
                                                      const __grid_constant__ DenTailP w) {
  __shared__ float4 sf[PRE ? 1 : 8][DT + 2];
  __shared__ float4 s0[4][DT];
  __shared__ float4 s1[2][DT - 2];
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * DT_OUT;
  const int tid = threadIdx.x;
  if (PRE) {
    // td0 output rows t0-2 .. t0+DT-3 from the conv engine (already LeakyReLU'd; zero outside [0,T))
    const int t = t0 - 2 + tid;
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.f;
    if (t >= 0 && t < T) {
      float lo[8], hi[8];
      unpack_half8(*reinterpret_cast<const uint4*>(h1 + act_off(h_bs, h_Tp, b, 0, t)), lo);
      unpack_half8(*reinterpret_cast<const uint4*>(h1 + act_off(h_bs, h_Tp, b, 1, t)), hi);
#pragma unroll
      for (int i = 0; i < 8; ++i) { v[i] = lo[i]; v[8 + i] = hi[i]; }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) s0[c][tid] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
  }
  // f tile: rows t0-3 .. t0+DT-2
  if (!PRE)
  for (int i = tid; i < 4 * (DT + 2); i += DT) {
    const int c = i / (DT + 2), r = i % (DT + 2);   // c: 8-channel chunk of the H8 input
    const int t = t0 - 3 + r;
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (t >= 0 && t < T) unpack_half8(*reinterpret_cast<const uint4*>(fin + act_off(f_bs, f_Tp, b, c, t)), v);
    sf[2 * c][r] = make_float4(v[0], v[1], v[2], v[3]);
    sf[2 * c + 1][r] = make_float4(v[4], v[5], v[6], v[7]);
  }
  __syncthreads();
  // td0: 32 -> 16 at rows t0-2 .. t0+DT-3 (local r in [0, DT)), input rows r..r+2 of sf
  if (!PRE) {
    const int r = tid;
    const int t = t0 - 2 + r;
    float acc[16];
#pragma unroll
    for (int o = 0; o < 16; ++o) acc[o] = w.b0[o];
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float4 v = sf[c][r + j];
#pragma unroll
        for (int o = 0; o < 16; ++o)
          acc[o] = fmaf(v.x, w.w0[j][4 * c][o], fmaf(v.y, w.w0[j][4 * c + 1][o], fmaf(v.z, w.w0[j][4 * c + 2][o], fmaf(v.w, w.w0[j][4 * c + 3][o], acc[o]))));
      }
    const bool ok = (t >= 0 && t < T);
#pragma unroll
    for (int o = 0; o < 16; ++o) acc[o] = ok ? (acc[o] > 0.f ? acc[o] : LRELU_SLOPE * acc[o]) : 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) s0[c][r] = make_float4(acc[4 * c], acc[4 * c + 1], acc[4 * c + 2], acc[4 * c + 3]);
  }
  __syncthreads();
  // td1: 16 -> 8 at rows t0-1 .. t0+DT-4 (local r in [0, DT-2))
  if (tid < DT - 2) {
    const int r = tid;
    const int t = t0 - 1 + r;
    // two output channels per FFMA2 (weight pair = one 8-byte constant-bank operand, input broadcast); per channel the same
    // accumulation order as the scalar form in the PRE = false branch above (bias, then per tap and 4-channel group w, z, y, x)
    unsigned long long acc2[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) acc2[o] = f2_pack(w.b1[2 * o], w.b1[2 * o + 1]);
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float4 v = s0[c][r + j];
        const float vin[4] = {v.w, v.z, v.y, v.x};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const unsigned long long vv = f2_pack(vin[k], vin[k]);
#pragma unroll
          for (int o = 0; o < 4; ++o) {
            const unsigned long long ww = f2_pack(w.w1[j][4 * c + 3 - k][2 * o], w.w1[j][4 * c + 3 - k][2 * o + 1]);
            asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc2[o]) : "l"(vv), "l"(ww));
          }
        }
      }
    float acc[8];
#pragma unroll
    for (int o = 0; o < 4; ++o) f2_unpack(acc2[o], acc[2 * o], acc[2 * o + 1]);
    const bool ok = (t >= 0 && t < T);
#pragma unroll
    for (int o = 0; o < 8; ++o) acc[o] = ok ? (acc[o] > 0.f ? acc[o] : LRELU_SLOPE * acc[o]) : 0.f;
    s1[0][r] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    s1[1][r] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  }
  __syncthreads();
  const int t = t0 + tid;
  if (tid >= DT_OUT || t >= T) return;
  // td2: 8 -> 1, sigmoid
  float m = w.b2;
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const float4 a0 = s1[0][tid + j], a1 = s1[1][tid + j];
    m += a0.x * w.w2[j][0] + a0.y * w.w2[j][1] + a0.z * w.w2[j][2] + a0.w * w.w2[j][3] + a1.x * w.w2[j][4] + a1.y * w.w2[j][5] +
         a1.z * w.w2[j][6] + a1.w * w.w2[j][7];
  }
  const float mt = 1.f / (1.f + expf(-m));
  // final 1x1 conv
  float yv = w.bf;
  if (PRE) {   // this thread's own row of f, straight from global memory
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float v[8];
      unpack_half8(*reinterpret_cast<const uint4*>(fin + act_off(f_bs, f_Tp, b, c, t)), v);
#pragma unroll
      for (int i = 0; i < 8; ++i) yv += v[i] * w.wf[8 * c + i];
    }
  } else {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float4 v = sf[c][tid + 3];
      yv += v.x * w.wf[4 * c] + v.y * w.wf[4 * c + 1] + v.z * w.wf[4 * c + 2] + v.w * w.wf[4 * c + 3];
    }
  }
  // analytic impulse mask from the raw input
  const float* xb = x + (long long)b * T;
  float xs[8];  // x[t-2 .. t+5)
#pragma unroll
  for (int i = 0; i < 7; ++i) {
    const int ti = t - 2 + i;
    xs[i] = (ti >= 0 && ti < T) ? __ldg(xb + ti) : 0.f;
  }
  float box = 0.f;
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const int u = t - 2 + i;
    if (u < 0 || u >= T) continue;
    const float d1u = (u < T - 1) ? fabsf(xs[i + 1] - xs[i]) : 0.f;
    const float d1n = (u + 1 < T - 1) ? fabsf(xs[i + 2] - xs[i + 1]) : 0.f;
    const float d2u = (u < T - 1) ? fabsf(d1n - d1u) : 0.f;
    box += (d2u * 2.0f + d1u + fabsf(xs[i]) * 0.5f) / 3.5f * 0.2f;
  }
  const float mi = fminf(fmaxf(box, 0.f), 1.f);
  y[(long long)b * T + t] = yv * (1.0f - fmaxf(mt, mi) * 0.9f);
}

int launch_den_tail(const Act& f, const Act* h1, const float* x, float* y, int B, int T, const DenTailP& w, cudaStream_t stream) {
  dim3 grid((T + DT_OUT - 1) / DT_OUT, B);
  if (h1 != nullptr)
    den_tail_kernel<true><<<grid, DT, 0, stream>>>(f.h(), f.bs, f.Tp, h1->h(), h1->bs, h1->Tp, x, y, T, w);
  else
    den_tail_kernel<false><<<grid, DT, 0, stream>>>(f.h(), f.bs, f.Tp, nullptr, 0, 0, x, y, T, w);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

// ============================================================================ normalize
// audio_processing.py:58-87.  Pass 1: per-block sum(x^2) and max|x|; pass 2: every block
// folds the (<= NORM_BLOCKS) partials in fp64, derives the gain on the device, scales.
constexpr int NORM_BLOCKS = 592;  // 4 per SM
constexpr int NORM_THREADS = 256;

__global__ void __launch_bounds__(NORM_THREADS) norm_reduce_kernel(const float* __restrict__ x, long long n, float* partial) {
  float ss = 0.f, mx = 0.f;
  const long long n4 = n >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = x4[i];
    ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    mx = fmaxf(mx, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = x[i];
    ss += v * v;
    mx = fmaxf(mx, fabsf(v));
  }
  __shared__ float s_ss[NORM_THREADS / 32], s_mx[NORM_THREADS / 32];
  for (int o = 16; o > 0; o >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { s_ss[threadIdx.x >> 5] = ss; s_mx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < NORM_THREADS / 32; ++i) { ss += s_ss[i]; mx = fmaxf(mx, s_mx[i]); }
    partial[2 * blockIdx.x] = ss;
    partial[2 * blockIdx.x + 1] = mx;
  }
}

__global__ void __launch_bounds__(NORM_THREADS) norm_scale_kernel(float* __restrict__ x, long long n, const float* __restrict__ partial,
                                                                  int nparts, float target_rms) {
  __shared__ double s_ss[NORM_THREADS / 32];
  __shared__ float s_mx[NORM_THREADS / 32];
  __shared__ float s_gain, s_peak;
  double ss = 0.0;
  float mx = 0.f;
  for (int i = threadIdx.x; i < nparts; i += blockDim.x) { ss += (double)partial[2 * i]; mx = fmaxf(mx, partial[2 * i + 1]); }
  for (int o = 16; o > 0; o >>= 1) {
    ss += __shfl_xor_sync(0xffffffffu, ss, o);
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { s_ss[threadIdx.x >> 5] = ss; s_mx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < NORM_THREADS / 32; ++i) { ss += s_ss[i]; mx = fmaxf(mx, s_mx[i]); }
    const float rms = (float)sqrt(ss / (double)n);
    float gain = 0.f, peak = 1.f;          // gain 0 => leave untouched (rms == 0 branch, :72)
    if (rms != 0.f) {
      gain = (1.0f / rms) * target_rms;     // torch evaluates `float / tensor` as reciprocal * float
      const float pk = mx * gain;           // == max|x*gain| because rounding is monotonic
      if (pk > 1.0f) peak = pk;             // :84-85
    }
    s_gain = gain;
    s_peak = peak;
  }
  __syncthreads();
  const float gain = s_gain, peak = s_peak;
  if (gain == 0.f) return;
  const bool limit = peak != 1.f;
  const long long n4 = n >> 2;
  float4* x4 = reinterpret_cast<float4*>(x);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 v = x4[i];
    v.x *= gain; v.y *= gain; v.z *= gain; v.w *= gain;
    if (limit) { v.x /= peak; v.y /= peak; v.z /= peak; v.w /= peak; }
    x4[i] = v;
  }
  for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float v = x[i] * gain;
    if (limit) v /= peak;
    x[i] = v;
  }
}

int launch_normalize(float* x, long long n, float target_db, float* scratch, cudaStream_t stream) {
  AR_CHECK(n > 0, AR_ERR_INVALID, "normalize: empty audio");
  AR_CHECK((reinterpret_cast<uintptr_t>(x) & 15) == 0, AR_ERR_INVALID, "normalize: audio must be 16-byte aligned");
  long long want = (n / 4 + NORM_THREADS - 1) / NORM_THREADS;
  int blocks = (int)(want < 1 ? 1 : (want > NORM_BLOCKS ? NORM_BLOCKS : want));
  norm_reduce_kernel<<<blocks, NORM_THREADS, 0, stream>>>(x, n, scratch);
  const float target_rms = (float)pow(10.0, (double)target_db / 20.0);
  norm_scale_kernel<<<blocks, NORM_THREADS, 0, stream>>>(x, n, scratch, blocks, target_rms);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

// ============================================================================ chunk split / overlap-add
__global__ void split_kernel(const float* __restrict__ audio, long long n, float* __restrict__ chunks, int first, int chunk_size, int hop) {
  const int ci = blockIdx.y;
  const long long start = (long long)(first + ci) * hop;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < chunk_size; j += gridDim.x * blockDim.x) {
    const long long s = start + j;
    chunks[(long long)ci * chunk_size + j] = (s < n) ? audio[s] : 0.f;  // zero-padded tail (trainer.py:660-665)
  }
}

int launch_split(const float* audio, long long n, float* chunks, int first, int count, int chunk_size, int overlap,
                 cudaStream_t stream) {
  if (count <= 0) return AR_OK;
  dim3 grid((chunk_size + 1023) / 1024 < 64 ? (chunk_size + 1023) / 1024 : 64, count);
  split_kernel<<<grid, 256, 0, stream>>>(audio, n, chunks, first, chunk_size, chunk_size - overlap);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

// out[c][p] = w*y_i[c][j] + (1-w)*y_{i-1}[c][j + r*hop] inside a cross-fade, y_i[c][j] elsewhere,
// with i = min(p / (r*hop), n_chunks-1), j = p - i*r*hop, w = (j+.5)/(r*overlap).
__global__ void ola_kernel(const float* __restrict__ y, float* __restrict__ out, long long n_out, int n_chunks, int channels,
                           int L /*rate*chunk*/, int H /*rate*hop*/, int V /*rate*overlap*/, float invV) {
  const int c = blockIdx.y;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n_out; p += (long long)gridDim.x * blockDim.x) {
    long long i = p / H;
    if (i > n_chunks - 1) i = n_chunks - 1;
    const long long j = p - i * H;
    float v = y[((long long)i * channels + c) * L + j];
    if (i > 0 && j < V) {
      const float w = ((float)j + 0.5f) * invV;
      const float prev = y[((long long)(i - 1) * channels + c) * L + (j + H)];
      v = v * w + prev * (1.0f - w);
    }
    out[(long long)c * n_out + p] = v;
  }
}

// Same gather, four output samples per thread: when the chunk length, the hop and the overlap at the output rate are all
// multiples of 4 (the default 2 x 44100 / 2 x 42048 / 2 x 2052 are) a 16-byte group of outputs lies in ONE chunk and entirely
// inside or outside its cross-fade, so it is one float4 load (two in a cross-fade) and one float4 store, with 32-bit index
// arithmetic (the scalar kernel spends its time in a 64-bit division per sample).  Bit-identical to the scalar kernel.
__global__ void __launch_bounds__(256) ola4_kernel(const float4* __restrict__ y, float4* __restrict__ out, unsigned n4 /*n_out / 4*/,
                                                   int n_chunks, int channels, unsigned L4, unsigned H4, unsigned V4, float invV) {
  const unsigned c = blockIdx.y;
  for (unsigned p = blockIdx.x * blockDim.x + threadIdx.x; p < n4; p += gridDim.x * blockDim.x) {
    unsigned i = p / H4;
    if (i > (unsigned)(n_chunks - 1)) i = n_chunks - 1;
    const unsigned j = p - i * H4;
    float4 v = __ldcs(y + ((size_t)i * channels + c) * L4 + j);          // read once: streaming
    if (i > 0 && j < V4) {
      const float4 q = __ldcs(y + ((size_t)(i - 1) * channels + c) * L4 + (j + H4));
      const float j0 = (float)(4 * j);
      const float w0 = (j0 + 0.5f) * invV, w1 = (j0 + 1.5f) * invV, w2 = (j0 + 2.5f) * invV, w3 = (j0 + 3.5f) * invV;
      v.x = v.x * w0 + q.x * (1.0f - w0);
      v.y = v.y * w1 + q.y * (1.0f - w1);
      v.z = v.z * w2 + q.z * (1.0f - w2);
      v.w = v.w * w3 + q.w * (1.0f - w3);
    }
    out[(size_t)c * n4 + p] = v;
  }
}

int launch_ola(const float* y, float* out, long long n, int n_chunks, int channels, int chunk_size, int overlap, int rate,
               cudaStream_t stream) {
  const long long n_out = n * rate;
  const int L = rate * chunk_size, H = rate * (chunk_size - overlap), V = rate * overlap;
  const float invV = V > 0 ? 1.0f / (float)V : 0.f;
  const bool vec = (L % 4 == 0) && (H % 4 == 0) && (V % 4 == 0) && (n_out % 4 == 0) && n_out < (1ll << 33) && V < (1 << 22) &&
                   ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(out)) & 15) == 0 &&
                   (long long)n_chunks * H / 4 + L / 4 < (1ll << 31);
  if (vec) {
    const long long want = (n_out / 4 + 255) / 256;
    dim3 grid((unsigned)(want > 2368 ? 2368 : want), channels);
    ola4_kernel<<<grid, 256, 0, stream>>>(reinterpret_cast<const float4*>(y), reinterpret_cast<float4*>(out), (unsigned)(n_out / 4),
                                          n_chunks, channels, L / 4, H / 4, V / 4, invV);
  } else {
    long long want = (n_out + 255) / 256;
    dim3 grid((unsigned)(want > 2368 ? 2368 : want), channels);
    ola_kernel<<<grid, 256, 0, stream>>>(y, out, n_out, n_chunks, channels, L, H, V, invV);
  }
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

// ============================================================================ window gather / kept-range scatter
// The lockstep whole-file-exact mode reads one window per file at a per-file offset of the stage-1 signals and writes one
// kept range per file back: one launch each way for all files of a step instead of one copy per file.
__global__ void gather_windows_kernel(const float* __restrict__ src, const long long* __restrict__ off, int W, float* __restrict__ dst) {
  const int b = blockIdx.y;
  const float* s = src + off[b];
  float* d = dst + (long long)b * W;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < W; j += gridDim.x * blockDim.x) d[j] = s[j];
}

__global__ void scatter_kept_kernel(const float* __restrict__ y, int W, const long long* __restrict__ dst_off,
                                    const int* __restrict__ lo, const int* __restrict__ len, float* __restrict__ out) {
  const int b = blockIdx.y, ch = blockIdx.z;
  const float* s = y + ((long long)b * 2 + ch) * W + lo[b];
  float* d = out + dst_off[2 * b + ch];
  const int n = len[b];
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) d[j] = s[j];
}

static int window_grid(int W) { return (W + 1023) / 1024 < 64 ? (W + 1023) / 1024 : 64; }

int launch_gather_windows(const float* src, long long src_len, const long long* offsets, int B, int W, float* dst, void* ws,
                          size_t ws_bytes, cudaStream_t stream) {
  AR_CHECK(src && offsets && dst && B >= 1 && W >= 1, AR_ERR_INVALID, "gather_windows: bad argument");
  AR_CHECK(ws != nullptr && ws_bytes >= (size_t)B * AR_WINDOW_IO_BYTES_PER_ITEM, AR_ERR_WORKSPACE, "gather_windows: workspace too small");
  for (int b = 0; b < B; ++b)
    AR_CHECK(offsets[b] >= 0 && offsets[b] + W <= src_len, AR_ERR_INVALID,
             "gather_windows: window " + std::to_string(b) + " at " + std::to_string(offsets[b]) + " leaves the source");
  long long* d_off = reinterpret_cast<long long*>(ws);
  AR_CUDA_OK(cudaMemcpyAsync(d_off, offsets, (size_t)B * sizeof(long long), cudaMemcpyHostToDevice, stream));
  gather_windows_kernel<<<dim3(window_grid(W), B), 256, 0, stream>>>(src, d_off, W, dst);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

int launch_scatter_kept(const float* y, int B, int W, const long long* dst_offsets, const int* lo, const int* len, float* out,
                        long long out_len, void* ws, size_t ws_bytes, cudaStream_t stream) {
  AR_CHECK(y && dst_offsets && lo && len && out && B >= 1 && W >= 1, AR_ERR_INVALID, "scatter_kept: bad argument");
  AR_CHECK(ws != nullptr && ws_bytes >= (size_t)B * AR_WINDOW_IO_BYTES_PER_ITEM, AR_ERR_WORKSPACE, "scatter_kept: workspace too small");
  int max_len = 0;
  for (int b = 0; b < B; ++b) {
    AR_CHECK(lo[b] >= 0 && len[b] >= 0 && lo[b] + len[b] <= W, AR_ERR_INVALID, "scatter_kept: kept range " + std::to_string(b) + " leaves its window");
    for (int ch = 0; ch < 2; ++ch)
      AR_CHECK(dst_offsets[2 * b + ch] >= 0 && dst_offsets[2 * b + ch] + len[b] <= out_len, AR_ERR_INVALID,
               "scatter_kept: kept range " + std::to_string(b) + " leaves the output");
    max_len = len[b] > max_len ? len[b] : max_len;
  }
  // one upload: [B][2] offsets, then lo[B], len[B]
  std::vector<char> stage((size_t)B * AR_WINDOW_IO_BYTES_PER_ITEM);
  memcpy(stage.data(), dst_offsets, (size_t)B * 16);
  memcpy(stage.data() + (size_t)B * 16, lo, (size_t)B * 4);
  memcpy(stage.data() + (size_t)B * 20, len, (size_t)B * 4);
  char* d = reinterpret_cast<char*>(ws);
  AR_CUDA_OK(cudaMemcpyAsync(d, stage.data(), stage.size(), cudaMemcpyHostToDevice, stream));   // pageable: staged on return
  if (max_len == 0) return AR_OK;
  scatter_kept_kernel<<<dim3(window_grid(max_len), B, 2), 256, 0, stream>>>(
      y, W, reinterpret_cast<const long long*>(d), reinterpret_cast<const int*>(d + (size_t)B * 16),
      reinterpret_cast<const int*>(d + (size_t)B * 20), out);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

// ============================================================================ layout converters (debug conv)
__global__ void plain_to_h8_kernel(const float* __restrict__ x, int C, int T, __half* __restrict__ out, long long bs, int Tp) {
  const int b = blockIdx.z, c8 = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  float v[8];
  for (int i = 0; i < 8; ++i) v[i] = x[((long long)b * C + c8 * 8 + i) * T + t];
  *reinterpret_cast<uint4*>(out + act_off(bs, Tp, b, c8, t)) = pack_half8(v);
}
// channel chunks [coff8, coff8 + gridDim.y) of an H8 (or, with tblock, time-blocked H8 of C8 chunks) tensor -> plain fp32
// [B][C][T] with C = 8 * gridDim.y
__global__ void h8_to_plain_kernel(const __half* __restrict__ in, long long bs, int Tp, int C8, int coff8, int tblock, int C, int T,
                                   float* __restrict__ y) {
  const int b = blockIdx.z, c8 = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const long long off = tblock ? act_off_tb(bs, C8, b, coff8 + c8, t) : act_off(bs, Tp, b, coff8 + c8, t);
  float v[8];
  unpack_half8(*reinterpret_cast<const uint4*>(in + off), v);
  for (int i = 0; i < 8; ++i) y[((long long)b * C + c8 * 8 + i) * T + t] = v[i];
}
int launch_plain_to_c4(const float* x, int B, int C, int T, const Act& out, cudaStream_t stream) {
  dim3 grid((T + 127) / 128, C / 8, B);
  plain_to_h8_kernel<<<grid, 128, 0, stream>>>(x, C, T, out.h(), out.bs, out.Tp);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}
int launch_c4_to_plain(const Act& in, int B, int C, int T, float* y, cudaStream_t stream) {
  dim3 grid((T + 127) / 128, C / 8, B);
  h8_to_plain_kernel<<<grid, 128, 0, stream>>>(in.h(), in.bs, in.Tp, in.C / 8, 0, 0, C, T, y);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}
int launch_audit_tap(const Act& a, int B, int coff8, int nch8, int T, int tblock, float* y, cudaStream_t stream) {
  dim3 grid((T + 127) / 128, nch8, B);
  h8_to_plain_kernel<<<grid, 128, 0, stream>>>(a.h(), a.bs, a.Tp, a.C / 8, coff8, tblock, nch8 * 8, T, y);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

// ----------------------------------------------------------------------------- dynamic-range audit
// max |value| over the valid rows [0,T) of an H8 (or time-blocked H8) activation tensor, folded into *slot with an
// atomic max on the float's bit pattern (non-negative floats order like unsigned integers).  fp16 storage saturates at
// +-65504: a layer whose maximum reaches that value has clipped (ar_model_audit_*).
__global__ void __launch_bounds__(256) audit_kernel(const __half* a, long long bs, int Tp, int C8, int coff8, int T, int tblock, unsigned int* slot) {
  const int b = blockIdx.z, ch = coff8 + blockIdx.y;
  float m = 0.f;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < T; t += gridDim.x * blockDim.x) {
    const long long off = tblock ? act_off_tb(bs, C8, b, ch, t) : act_off(bs, Tp, b, ch, t);
    float v[8];
    unpack_half8(*reinterpret_cast<const uint4*>(a + off), v);
#pragma unroll
    for (int i = 0; i < 8; ++i) m = fmaxf(m, fabsf(v[i]));   // fmaxf drops a NaN operand: NaNs are caught by the finite check of the output
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(slot, __float_as_uint(m));
}

int launch_audit(const Act& a, int B, int coff8, int nch8, int T, int tblock, unsigned int* slot, cudaStream_t stream) {
  int gx = (T + 255) / 256;
  if (gx > 64) gx = 64;
  dim3 grid(gx, nch8, B);
  audit_kernel<<<grid, 256, 0, stream>>>(a.h(), a.bs, a.Tp, a.C / 8, coff8, T, tblock, slot);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

}  // namespace ar
