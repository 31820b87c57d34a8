// FLAC encoder on the GPU (RFC 9639): the torchaudio.save of a .flac path (src/utils/audio_processing.py:45-55).  Input:
// planar fp32 [channels][n] on the device; output: the frame section of one stream (the caller writes `fLaC` and
// STREAMINFO in front) and the interleaved little-endian PCM bytes the STREAMINFO MD5 is taken over.
//
// Every choice is defined and integer-only, so tests/flac_encode_ref.py::encode_search restates it byte for byte:
//   - fixed blocking, frames coded by frame number, a short last frame;
//   - per coded channel: wasted bits (trailing zeros of the OR of the block, capped at depth - 1), then the fewest exact
//     bits of CONSTANT (all samples equal), FIXED orders 0..4 (order <= block size) and VERBATIM, ties to that order;
//   - FIXED residuals coded with an exact search over RICE (4-bit k <= 14) and RICE2 (5-bit k <= 30) and partition
//     orders 0..8 (bs % 2^p == 0, (bs >> p) >= order): Σ(u >> k) for every k on the finest leaves, summed up the tree;
//     ties to the smaller method, partition order, k.  Escape codes are never written (u < 2^30, so k = 30 suffices);
//   - two channels: the cheapest of independent / left-side / side-right / mid-side, ties to the lower code.
// Kernels:
//   1. quantise : q = rint_even(clamp(x, -1, 1) * (2^(bps-1) - 1)) (fp32 multiply, no FMA; NaN -> 0) as int32 planar, and
//                 the PCM bytes for the MD5 (HBM-bound).
//   2. analyse  : one CTA per frame: the search above, one signal at a time in shared memory; writes a descriptor per
//                 coded channel (type, order, wasted bits, method, partition order, exact bits) and the k of each partition.
//   3. write    : one CTA per frame into a zeroed shared-memory buffer: header and CRC-8, subframe fields, residual codes at
//                 bit positions from a block prefix sum of code lengths (unary zeros are the buffer's zeros, so a code
//                 writes its stop bit and k low bits: at most two atomicOr on 32-bit words), padding, a parallel CRC-16.
//                 Checks the bits written against the descriptor, then copies the frame into its own slot.
//   4. finish / gather : exclusive scan of frame bytes (one CTA; also min / max frame bytes and the first frame whose
//                 status is not OK), then every slot copied to its offset in the contiguous output.
// Fault safety: a slot holds the VERBATIM bound of a full block (header 16 + Σ_c ceil((8 + bs·depth_c)/8) + CRC 2,
// rounded up to 16 bytes) and every candidate includes VERBATIM, so no frame is larger; still every shared and global
// store is guarded against its buffer's end and every input load against n, and a frame that does not write exactly the
// bits it was sized for is reported (AR_ERR_INVALID), never truncated silently.
#include <climits>
#include <cstdio>

#include "ar_common.cuh"
#include "flac_common.cuh"

namespace ar {

namespace {

constexpr int ET = 256;              // threads per CTA of the analyse / write kernels
constexpr int MAX_BLOCK = 4608;      // the largest block of the streamable subset at every rate
constexpr int MAX_RATE = 655350;
constexpr int MAX_LEAVES = 256;      // partition order <= 8
constexpr int NK = 31;               // Rice parameters 0..30
constexpr int SROW = 33;             // leaf-sum row stride (64-bit words): odd, so rows spread over the banks
constexpr int HEADER_MAX = 16;       // sync 2 + codes 2 + frame number <= 6 + block size <= 2 + rate <= 2 + CRC-8 1
constexpr int FIN_THREADS = 1024;

enum EncStatus { ST_OK = 0, ST_BITS = 1, ST_OVERFLOW = 2 };

struct EncParams {
  long long n, frames;
  int channels, bps, block, sample_rate, kcap;
};

struct SubDesc {             // one coded channel of one frame
  long long bits;            // exact subframe bits
  int type;                  // 0 CONSTANT, 1 VERBATIM, 8 + order FIXED
  int wasted, method, porder;
};

struct FrameStat {
  long long wrote, sized;    // bits the writer produced / the descriptors promised (header and subframes)
  int bytes, status;
};

struct Summary {
  long long total, bad_frame, wrote, sized;
  int min_bytes, max_bytes, status, pad;
};

__host__ __device__ inline int leaf_order(int bs) {    // the largest p <= 8 with bs % 2^p == 0
  int p = 0;
  while (p < 8 && bs % (2 << p) == 0) ++p;
  return p;
}

__host__ __device__ inline long long slot_bytes(int block, int channels, int bps) {
  long long b = HEADER_MAX + 2;
  for (int c = 0; c < channels; ++c) b += (8 + (long long)block * (bps + (channels == 2 && c == 1)) + 7) / 8;
  return (b + 15) & ~15LL;
}

// Frame header with its CRC-8 into h (<= HEADER_MAX bytes); returns its length.  Codes as tests/flac_encode_ref.py.
__device__ int frame_header(unsigned char* h, long long number, int bs, int rate, int assign, int bps) {
  int bcode;
  switch (bs) {
    case 192: bcode = 1; break;
    case 576: bcode = 2; break;
    case 1152: bcode = 3; break;
    case 2304: bcode = 4; break;
    case 4608: bcode = 5; break;
    case 256: bcode = 8; break;
    case 512: bcode = 9; break;
    case 1024: bcode = 10; break;
    case 2048: bcode = 11; break;
    case 4096: bcode = 12; break;
    default: bcode = bs <= 256 ? 6 : 7; break;
  }
  int rcode;
  switch (rate) {
    case 88200: rcode = 1; break;
    case 176400: rcode = 2; break;
    case 192000: rcode = 3; break;
    case 8000: rcode = 4; break;
    case 16000: rcode = 5; break;
    case 22050: rcode = 6; break;
    case 24000: rcode = 7; break;
    case 32000: rcode = 8; break;
    case 44100: rcode = 9; break;
    case 48000: rcode = 10; break;
    case 96000: rcode = 11; break;
    default:
      rcode = (rate % 1000 == 0 && rate / 1000 < 256) ? 12 : rate < 65536 ? 13 : (rate % 10 == 0 && rate / 10 < 65536) ? 14 : 0;
  }
  int i = 0;
  h[i++] = 0xFF;
  h[i++] = 0xF8;
  h[i++] = (unsigned char)((bcode << 4) | rcode);
  h[i++] = (unsigned char)((assign << 4) | ((bps == 16 ? 4 : 6) << 1));
  if (number < 0x80) {
    h[i++] = (unsigned char)number;
  } else {                                                   // UTF-8-style: nb bytes hold 5 * nb + 1 bits
    int nb = 2;
    while (number >= (1LL << (5 * nb + 1))) ++nb;
    h[i++] = (unsigned char)(((0xFF00 >> nb) & 0xFF) | (number >> (6 * (nb - 1))));
    for (int j = nb - 2; j >= 0; --j) h[i++] = (unsigned char)(0x80 | ((number >> (6 * j)) & 0x3F));
  }
  if (bcode == 6) h[i++] = (unsigned char)(bs - 1);
  if (bcode == 7) { h[i++] = (unsigned char)((bs - 1) >> 8); h[i++] = (unsigned char)(bs - 1); }
  if (rcode == 12) h[i++] = (unsigned char)(rate / 1000);
  if (rcode == 13) { h[i++] = (unsigned char)(rate >> 8); h[i++] = (unsigned char)rate; }
  if (rcode == 14) { h[i++] = (unsigned char)((rate / 10) >> 8); h[i++] = (unsigned char)(rate / 10); }
  h[i] = (unsigned char)crc8_bytes(h, i);
  return i + 1;
}

// Signal `sig` at absolute sample `at` (< n): channel sig, or for two channels L, R, S = L - R, M = (L + R) >> 1.
__device__ __forceinline__ int load_signal(const int* __restrict__ q, long long n, int channels, int sig, long long at) {
  if (channels != 2 || sig < 2) return q[sig * n + at];
  const int l = q[at], r = q[n + at];
  return sig == 2 ? l - r : (l + r) >> 1;
}

// Signal of coded channel c under channel assignment `assign` (1 independent, 8 left/side, 9 side/right, 10 mid/side).
__device__ __forceinline__ int coded_signal(int assign, int channels, int c) {
  if (channels != 2 || assign == 1) return c;
  if (assign == 8) return c == 0 ? 0 : 2;
  if (assign == 9) return c == 0 ? 2 : 1;
  return c == 0 ? 3 : 2;
}

// FIXED order-o residual of s[i] (i >= o): the o-th difference.  |r| < 2^28 for 25-bit samples.
__device__ __forceinline__ int fixed_residual(const int* s, int i, int o) {
  switch (o) {
    case 0: return s[i];
    case 1: return s[i] - s[i - 1];
    case 2: return s[i] - 2 * s[i - 1] + s[i - 2];
    case 3: return s[i] - 3 * (s[i - 1] - s[i - 2]) - s[i - 3];
    default: return s[i] - 4 * (s[i - 1] + s[i - 3]) + 6 * s[i - 2] + s[i - 4];
  }
}

__device__ __forceinline__ unsigned zigzag(int r) { return ((unsigned)r << 1) ^ (unsigned)(r >> 31); }

// Sum over the CTA; every thread receives the total.  `red` holds ET / 32 entries.
__device__ __forceinline__ long long block_sum(long long v, long long* red) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  long long t = 0;
  for (int w = 0; w < ET / 32; ++w) t += red[w];
  return t;
}

// Exclusive prefix sum over the CTA in thread order; *total receives the sum.
__device__ __forceinline__ long long block_exclusive_scan(long long v, long long* red, long long* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long incl = v;
  for (int o = 1; o < 32; o <<= 1) {
    const long long y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  __syncthreads();
  if (lane == 31) red[warp] = incl;
  __syncthreads();
  long long before = 0, t = 0;
  for (int w = 0; w < ET / 32; ++w) {
    const long long r = red[w];
    if (w < warp) before += r;
    t += r;
  }
  *total = t;
  return before + incl - v;
}

__global__ void flac_enc_quantise_kernel(const float* __restrict__ x, long long n, int channels, int bps, int* __restrict__ q,
                                         unsigned char* __restrict__ pcm) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float scale = (float)((1 << (bps - 1)) - 1);
  const int width = bps >> 3;
  for (int c = 0; c < channels; ++c) {
    const float v = x[c * n + i];
    const int s = isnan(v) ? 0 : __float2int_rn(__fmul_rn(fminf(fmaxf(v, -1.0f), 1.0f), scale));
    q[c * n + i] = s;
    unsigned char* o = pcm + (i * channels + c) * width;
    o[0] = (unsigned char)s;
    o[1] = (unsigned char)(s >> 8);
    if (width == 3) o[2] = (unsigned char)(s >> 16);
  }
}

// Dynamic shared memory of the analyse kernel: leaf sums [MAX_LEAVES][SROW] u64, samples and zigzag residuals [block]
// each, best k per (method, level, partition) and per signal.
size_t analyse_smem(int block) {
  return sizeof(unsigned long long) * MAX_LEAVES * SROW + 2 * sizeof(int) * (size_t)block + 2 * 9 * MAX_LEAVES + 8 * MAX_LEAVES;
}

__global__ void __launch_bounds__(ET) flac_enc_analyse_kernel(const int* __restrict__ q, EncParams ep, SubDesc* __restrict__ desc,
                                                              unsigned char* __restrict__ kout, int* __restrict__ assign_out) {
  extern __shared__ __align__(16) unsigned char smem[];
  unsigned long long* S = reinterpret_cast<unsigned long long*>(smem);                 // [leaf][k], row stride SROW
  int* s = reinterpret_cast<int*>(S + MAX_LEAVES * SROW);                              // [block] samples >> wasted
  unsigned* u = reinterpret_cast<unsigned*>(s + ep.block);                              // [block] zigzag residuals
  unsigned char* kb = reinterpret_cast<unsigned char*>(u + ep.block);                   // [2][9][MAX_LEAVES]
  unsigned char* sigk = kb + 2 * 9 * MAX_LEAVES;                                        // [8][MAX_LEAVES]
  __shared__ SubDesc sd[8];
  __shared__ long long red[ET / 32];
  __shared__ long long tot[2][9];
  __shared__ int s_or, s_neq;

  const long long f = blockIdx.x;
  const long long first = f * ep.block;
  const int bs = (int)min((long long)ep.block, ep.n - first);
  const int P = leaf_order(bs), leaves = 1 << P, lsize = bs >> P;
  const int nsig = ep.channels == 2 ? 4 : ep.channels;
  const int tid = threadIdx.x;

  for (int sig = 0; sig < nsig; ++sig) {
    const int depth = ep.bps + (ep.channels == 2 && sig == 2);
    if (tid == 0) { s_or = 0; s_neq = 0; }
    __syncthreads();
    int orr = 0;
    for (int i = tid; i < bs; i += ET) {
      const int v = load_signal(q, ep.n, ep.channels, sig, first + i);
      s[i] = v;
      orr |= v;
    }
    atomicOr(&s_or, orr);
    __syncthreads();
    const int v0 = s[0];
    const int w = s_or == 0 ? 0 : min(__ffs(s_or) - 1, depth - 1);
    __syncthreads();
    int neq = 0;
    for (int i = tid; i < bs; i += ET) {
      const int v = s[i];
      neq |= v != v0;
      s[i] = v >> w;
    }
    if (neq) atomicOr(&s_neq, 1);
    __syncthreads();
    const int ed = depth - w, head = 8 + w;
    long long best = s_neq ? LLONG_MAX : head + ed;
    int type = 0, method = 0, porder = 0;

    for (int o = 0; o <= 4 && o <= bs; ++o) {
      for (int i = tid; i < bs; i += ET) u[i] = i < o ? 0u : zigzag(fixed_residual(s, i, o));
      __syncthreads();
      for (int c = tid; c < leaves * NK; c += ET) {                      // k fastest: a warp reads one or two leaves
        const int l = c / NK, k = c - l * NK;
        unsigned long long acc = 0;
        for (int t = 0; t < lsize; ++t) acc += u[l * lsize + t] >> k;
        S[l * SROW + k] = acc;
      }
      __syncthreads();
      for (int p = P; p >= 0; --p) {
        if ((bs >> p) >= o) {                                             // a partition holds at least the warm-up
          long long b4 = 0, b5 = 0;
          if (tid < (1 << p)) {
            const unsigned long long* row = S + (long long)(tid << (P - p)) * SROW;
            const long long cnt = (bs >> p) - (tid == 0 ? o : 0);
            long long m4 = LLONG_MAX, m5 = LLONG_MAX;
            int k4 = 0, k5 = 0;
            for (int k = 0; k < NK; ++k) {
              const long long cost = (long long)row[k] + cnt * (k + 1);
              if (k <= 14 && cost < m4) { m4 = cost; k4 = k; }
              if (cost < m5) { m5 = cost; k5 = k; }
            }
            kb[(0 * 9 + p) * MAX_LEAVES + tid] = (unsigned char)k4;
            kb[(1 * 9 + p) * MAX_LEAVES + tid] = (unsigned char)k5;
            b4 = m4 + 4;
            b5 = m5 + 5;
          }
          b4 = block_sum(b4, red);
          b5 = block_sum(b5, red);
          if (tid == 0) { tot[0][p] = 6 + b4; tot[1][p] = 6 + b5; }
        } else if (tid == 0) {
          tot[0][p] = tot[1][p] = LLONG_MAX;
        }
        if (p > 0) {                                                      // in-place upsweep to level p - 1
          const int half = 1 << (p - 1), step = 1 << (P - p);
          for (int c = tid; c < half * NK; c += ET) {
            const int j = c / NK, k = c - j * NK;
            S[(long long)(2 * j * step) * SROW + k] += S[(long long)((2 * j + 1) * step) * SROW + k];
          }
        }
        __syncthreads();
      }
      int bm = -1, bp = 0;                                                // every thread takes the same decision
      long long bt = LLONG_MAX;
      for (int m = 0; m < 2; ++m)
        for (int p = 0; p <= P; ++p)
          if (tot[m][p] < bt) { bt = tot[m][p]; bm = m; bp = p; }
      if (bm >= 0 && head + (long long)o * ed + bt < best) {
        best = head + (long long)o * ed + bt;
        type = 8 + o;
        method = bm;
        porder = bp;
        for (int j = tid; j < (1 << bp); j += ET) sigk[sig * MAX_LEAVES + j] = kb[(bm * 9 + bp) * MAX_LEAVES + j];
      }
      __syncthreads();
    }
    if (head + (long long)bs * ed < best) { best = head + (long long)bs * ed; type = 1; }
    if (tid == 0) sd[sig] = SubDesc{best, type, w, method, porder};
    __syncthreads();
  }

  int assign = ep.channels - 1;
  if (ep.channels == 2) {
    const long long c1 = sd[0].bits + sd[1].bits, c8 = sd[0].bits + sd[2].bits, c9 = sd[2].bits + sd[1].bits,
                    c10 = sd[3].bits + sd[2].bits;
    long long b = c1;
    if (c8 < b) { b = c8; assign = 8; }
    if (c9 < b) { b = c9; assign = 9; }
    if (c10 < b) { assign = 10; }
  }
  for (int c = 0; c < ep.channels; ++c) {
    const int sig = coded_signal(assign, ep.channels, c);
    const SubDesc d = sd[sig];
    const long long at = f * ep.channels + c;
    if (tid == 0) desc[at] = d;
    if (d.type >= 8)
      for (int j = tid; j < (1 << d.porder) && j < ep.kcap; j += ET) kout[at * ep.kcap + j] = sigk[sig * MAX_LEAVES + j];
  }
  if (tid == 0) assign_out[f] = assign;
}

// OR `width` (1..32) bits of v (< 2^width) into the MSB-first bit stream buf[nwords] at bit `pos`.
__device__ __forceinline__ void put_bits(unsigned* buf, long long nwords, long long pos, int width, unsigned v, int* overflow) {
  if (width <= 0) return;
  const long long w0 = pos >> 5;
  const int sh = (int)(pos & 31);
  if (pos < 0 || ((pos + width - 1) >> 5) >= nwords) { *overflow = 1; return; }
  if (sh + width <= 32) {
    atomicOr(&buf[w0], v << (32 - sh - width));
  } else {
    atomicOr(&buf[w0], v >> (sh + width - 32));
    atomicOr(&buf[w0 + 1], v << (64 - sh - width));
  }
}

__device__ __forceinline__ unsigned buf_byte(const unsigned* buf, long long b) { return (buf[b >> 2] >> (24 - 8 * (b & 3))) & 0xFF; }

__device__ unsigned gf16_mul(unsigned a, unsigned b) {                  // a * b mod (x^16 + x^15 + x^2 + 1)
  unsigned r = 0;
  for (int i = 15; i >= 0; --i) {
    r <<= 1;
    if (r & 0x10000) r ^= 0x18005;
    if ((b >> i) & 1) r ^= a;
  }
  return r;
}

// CRC-16 of bytes followed by `nbytes` zero bytes, from the CRC of the bytes: crc * x^(8 nbytes) mod P.  With initial
// value 0 the CRC is linear, so the CRC of a frame is the XOR of its chunks' CRCs shifted by the bytes after each chunk.
__device__ unsigned crc16_shift(unsigned crc, long long nbytes) {
  unsigned pw = 0x100;                                                   // x^8
  for (; nbytes; nbytes >>= 1) {
    if (nbytes & 1) crc = gf16_mul(crc, pw);
    pw = gf16_mul(pw, pw);
  }
  return crc;
}

__global__ void __launch_bounds__(ET) flac_enc_write_kernel(const int* __restrict__ q, EncParams ep, const SubDesc* __restrict__ desc,
                                                            const unsigned char* __restrict__ kin, const int* __restrict__ assign_in,
                                                            unsigned char* __restrict__ slots, long long slot_cap,
                                                            FrameStat* __restrict__ stat) {
  extern __shared__ __align__(16) unsigned char smem[];
  const long long nwords = slot_cap >> 2;
  unsigned* buf = reinterpret_cast<unsigned*>(smem);                     // the frame, MSB-first within each word
  int* s = reinterpret_cast<int*>(buf + nwords);                         // [block] samples >> wasted
  __shared__ unsigned short crc_tab[256];
  __shared__ unsigned char hdr[HEADER_MAX];
  __shared__ long long red[ET / 32];
  __shared__ int s_hlen, s_overflow;

  const long long f = blockIdx.x;
  const long long first = f * ep.block;
  const int bs = (int)min((long long)ep.block, ep.n - first);
  const int assign = assign_in[f];
  const int tid = threadIdx.x;
  for (long long j = tid; j < nwords; j += ET) buf[j] = 0u;
  if (tid == 0) {
    s_hlen = frame_header(hdr, f, bs, ep.sample_rate, assign, ep.bps);
    s_overflow = 0;
  }
  crc16_table(crc_tab);                                                  // ends with a barrier
  if (tid < s_hlen) put_bits(buf, nwords, tid * 8, 8, hdr[tid], &s_overflow);
  long long pos = s_hlen * 8, sized = pos;
  bool bits_ok = true;

  for (int c = 0; c < ep.channels; ++c) {
    const SubDesc d = desc[f * ep.channels + c];
    const int sig = coded_signal(assign, ep.channels, c);
    const int depth = ep.bps + (ep.channels == 2 && sig == 2);
    const int w = d.wasted, ed = depth - w, head = 8 + w;
    const unsigned mask = (1u << ed) - 1u;
    for (int i = tid; i < bs; i += ET) s[i] = load_signal(q, ep.n, ep.channels, sig, first + i) >> w;
    __syncthreads();
    if (tid == 0) {
      put_bits(buf, nwords, pos, 8, (unsigned)((d.type << 1) | (w > 0)), &s_overflow);
      if (w > 0) put_bits(buf, nwords, pos + 8, w, 1u, &s_overflow);   // w - 1 zeros and a one
    }
    const long long p0 = pos + head;
    long long wrote;
    if (d.type == 0) {
      if (tid == 0) put_bits(buf, nwords, p0, ed, (unsigned)s[0] & mask, &s_overflow);
      wrote = head + ed;
    } else if (d.type == 1) {
      for (int i = tid; i < bs; i += ET) put_bits(buf, nwords, p0 + (long long)i * ed, ed, (unsigned)s[i] & mask, &s_overflow);
      wrote = head + (long long)bs * ed;
    } else {
      const int o = d.type - 8, pbits = 4 + d.method, ps = bs >> d.porder;
      const unsigned char* kc = kin + (f * ep.channels + c) * ep.kcap;
      if (tid < o) put_bits(buf, nwords, p0 + (long long)tid * ed, ed, (unsigned)s[tid] & mask, &s_overflow);
      const long long r0 = p0 + (long long)o * ed;
      if (tid == 0) {
        put_bits(buf, nwords, r0, 2, (unsigned)d.method, &s_overflow);
        put_bits(buf, nwords, r0 + 2, 4, (unsigned)d.porder, &s_overflow);
      }
      const int chunk = (bs + ET - 1) / ET;
      const int lo = min(bs, tid * chunk), hi = min(bs, lo + chunk);
      long long len = 0;
      for (int i = lo; i < hi; ++i) {
        const int k = kc[i / ps];
        if (i % ps == 0) len += pbits;
        if (i >= o) len += (zigzag(fixed_residual(s, i, o)) >> k) + 1 + k;
      }
      long long total;
      long long at = r0 + 6 + block_exclusive_scan(len, red, &total);
      for (int i = lo; i < hi; ++i) {
        const int k = kc[i / ps];
        if (i % ps == 0) { put_bits(buf, nwords, at, pbits, (unsigned)k, &s_overflow); at += pbits; }
        if (i >= o) {
          const unsigned uu = zigzag(fixed_residual(s, i, o));
          const long long zeros = uu >> k;
          put_bits(buf, nwords, at + zeros, k + 1, (1u << k) | (uu & ((1u << k) - 1u)), &s_overflow);
          at += zeros + 1 + k;
        }
      }
      wrote = head + (long long)o * ed + 6 + total;
    }
    bits_ok = bits_ok && wrote == d.bits;
    pos += wrote;
    sized += d.bits;
    __syncthreads();                                                     // s[] is reloaded for the next channel
  }

  // byte padding (the buffer is zero), then the CRC-16 of everything before it, in ET chunks
  const long long nbody = (pos + 7) >> 3;
  const long long chunk = (nbody + ET - 1) / ET;
  const long long lo = min(nbody, tid * chunk), hi = min(nbody, lo + chunk);
  unsigned crc = 0;
  for (long long b = lo; b < hi && (b >> 2) < nwords; ++b)
    crc = ((crc << 8) & 0xFFFF) ^ crc_tab[((crc >> 8) ^ buf_byte(buf, b)) & 0xFF];
  crc = crc16_shift(crc, nbody - hi);
  for (int o = 16; o; o >>= 1) crc ^= __shfl_xor_sync(0xffffffffu, crc, o);
  __syncthreads();
  if ((tid & 31) == 0) red[tid >> 5] = crc;
  __syncthreads();
  const long long bytes = nbody + 2;
  if (tid == 0) {
    unsigned all = 0;
    for (int wi = 0; wi < ET / 32; ++wi) all ^= (unsigned)red[wi];
    put_bits(buf, nwords, nbody * 8, 16, all, &s_overflow);
  }
  __syncthreads();
  const int status = s_overflow || bytes > slot_cap ? ST_OVERFLOW : bits_ok ? ST_OK : ST_BITS;
  unsigned char* slot = slots + f * slot_cap;
  for (long long j = tid; j < (bytes + 3) >> 2 && j < nwords; j += ET)
    reinterpret_cast<unsigned*>(slot)[j] = __byte_perm(buf[j], 0, 0x0123);
  if (tid == 0) stat[f] = FrameStat{pos, sized, status == ST_OK ? (int)bytes : 0, status};
}

// One CTA: exclusive scan of the frame bytes into offsets, the total, min / max frame bytes and the first frame whose
// status is not OK (fixed order: deterministic).
__global__ void __launch_bounds__(FIN_THREADS) flac_enc_finish_kernel(const FrameStat* __restrict__ stat, long long frames,
                                                                      long long* __restrict__ offsets, Summary* __restrict__ sum) {
  __shared__ long long part[FIN_THREADS], bad[FIN_THREADS];
  __shared__ int mins[FIN_THREADS], maxs[FIN_THREADS];
  const long long per = (frames + FIN_THREADS - 1) / FIN_THREADS;
  const long long lo = threadIdx.x * per, hi = min(frames, lo + per);
  long long t = 0, b = LLONG_MAX;
  int mn = INT_MAX, mx = 0;
  for (long long f = lo; f < hi; ++f) {
    const FrameStat e = stat[f];
    t += e.bytes;
    mn = min(mn, e.bytes);
    mx = max(mx, e.bytes);
    if (e.status != ST_OK && b == LLONG_MAX) b = f;
  }
  part[threadIdx.x] = t;
  bad[threadIdx.x] = b;
  mins[threadIdx.x] = mn;
  maxs[threadIdx.x] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    Summary r{0, LLONG_MAX, 0, 0, INT_MAX, 0, ST_OK, 0};
    for (int i = 0; i < FIN_THREADS; ++i) {
      const long long v = part[i];
      part[i] = r.total;
      r.total += v;
      r.min_bytes = min(r.min_bytes, mins[i]);
      r.max_bytes = max(r.max_bytes, maxs[i]);
      if (bad[i] < r.bad_frame) r.bad_frame = bad[i];
    }
    if (r.bad_frame != LLONG_MAX) {
      const FrameStat e = stat[r.bad_frame];
      r.wrote = e.wrote;
      r.sized = e.sized;
      r.status = e.status;
    }
    *sum = r;
  }
  __syncthreads();
  t = part[threadIdx.x];
  for (long long f = lo; f < hi; ++f) {
    offsets[f] = t;
    t += stat[f].bytes;
  }
}

__global__ void flac_enc_gather_kernel(const unsigned char* __restrict__ slots, long long slot_cap, const FrameStat* __restrict__ stat,
                                       const long long* __restrict__ offsets, unsigned char* __restrict__ out, long long out_cap) {
  const long long f = blockIdx.x;
  const long long nb = min((long long)stat[f].bytes, slot_cap), off = offsets[f];
  const unsigned char* slot = slots + f * slot_cap;
  for (long long b = threadIdx.x; b < nb; b += blockDim.x)
    if (off + b < out_cap) out[off + b] = slot[b];
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

struct EncLayout {
  long long frames, slot;
  int kcap;
  size_t q, desc, ks, assign, stat, offsets, sum, slots, bytes, out_capacity;
};

EncLayout enc_layout(int channels, long long n, int block, int bps) {
  EncLayout l;
  l.frames = (n + block - 1) / block;
  l.slot = slot_bytes(block, channels, bps);
  l.kcap = block < MAX_LEAVES ? block : MAX_LEAVES;                     // 2^porder <= min(bs, 256)
  size_t o = 0;
  l.q = o;       o += align256(sizeof(int) * (size_t)channels * (size_t)n);
  l.desc = o;    o += align256(sizeof(SubDesc) * (size_t)l.frames * channels);
  l.ks = o;      o += align256((size_t)l.frames * channels * l.kcap);
  l.assign = o;  o += align256(sizeof(int) * (size_t)l.frames);
  l.stat = o;    o += align256(sizeof(FrameStat) * (size_t)l.frames);
  l.offsets = o; o += align256(sizeof(long long) * (size_t)l.frames);
  l.sum = o;     o += align256(sizeof(Summary));
  l.slots = o;   o += align256((size_t)l.frames * (size_t)l.slot);
  l.bytes = o;
  l.out_capacity = (size_t)l.frames * (size_t)l.slot;
  return l;
}

int check_args(int channels, long long n, int block, int bps) {
  AR_CHECK(channels >= 1 && channels <= 8, AR_ERR_INVALID, "flac_encode: channels must be 1..8");
  AR_CHECK(bps == 16 || bps == 24, AR_ERR_INVALID, "flac_encode: bits per sample must be 16 or 24");
  AR_CHECK(block >= 16 && block <= MAX_BLOCK, AR_ERR_INVALID, "flac_encode: block size must be 16..4608");
  AR_CHECK(n >= 1 && n < (1LL << 36) && (n + block - 1) / block < (1LL << 31), AR_ERR_INVALID,
           "flac_encode: sample count must be 1..2^36 - 1 and at most 2^31 - 1 frames");
  return AR_OK;
}

}  // namespace

int flac_encode_workspace_bytes(int channels, long long n, int block_size, int bps, size_t* workspace, size_t* out_capacity) {
  AR_CHECK(workspace && out_capacity, AR_ERR_INVALID, "flac_encode_workspace_bytes: bad argument");
  AR_TRY(check_args(channels, n, block_size, bps));
  const EncLayout l = enc_layout(channels, n, block_size, bps);
  *workspace = l.bytes;
  *out_capacity = l.out_capacity;
  return AR_OK;
}

int flac_encode(const float* x, int channels, long long n, int bps, int sample_rate, int block_size, unsigned char* frames_out,
                size_t out_capacity, unsigned char* pcm_le_out, long long* frame_bytes_total, int* min_frame, int* max_frame,
                void* ws, size_t ws_bytes, cudaStream_t stream) {
  AR_TRY(check_args(channels, n, block_size, bps));
  AR_CHECK(x && frames_out && pcm_le_out && frame_bytes_total && min_frame && max_frame, AR_ERR_INVALID,
           "flac_encode: bad argument");
  AR_CHECK(sample_rate >= 1 && sample_rate <= MAX_RATE, AR_ERR_INVALID, "flac_encode: sample rate must be 1..655350 Hz");
  const EncLayout l = enc_layout(channels, n, block_size, bps);
  AR_CHECK(out_capacity >= l.out_capacity, AR_ERR_INVALID, "flac_encode: output capacity too small (ar_flac_encode_workspace_bytes)");
  AR_CHECK(ws && ws_bytes >= l.bytes, AR_ERR_WORKSPACE, "flac_encode: workspace too small (ar_flac_encode_workspace_bytes)");
  char* w = static_cast<char*>(ws);
  int* q = reinterpret_cast<int*>(w + l.q);
  SubDesc* desc = reinterpret_cast<SubDesc*>(w + l.desc);
  unsigned char* ks = reinterpret_cast<unsigned char*>(w + l.ks);
  int* assign = reinterpret_cast<int*>(w + l.assign);
  FrameStat* stat = reinterpret_cast<FrameStat*>(w + l.stat);
  long long* offsets = reinterpret_cast<long long*>(w + l.offsets);
  Summary* sum_dev = reinterpret_cast<Summary*>(w + l.sum);
  unsigned char* slots = reinterpret_cast<unsigned char*>(w + l.slots);
  const EncParams ep{n, l.frames, channels, bps, block_size, sample_rate, l.kcap};

  const size_t a_smem = analyse_smem(block_size);
  const size_t w_smem = (size_t)l.slot + sizeof(int) * (size_t)block_size;
  AR_CUDA_OK(cudaFuncSetAttribute(flac_enc_analyse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)a_smem));
  AR_CUDA_OK(cudaFuncSetAttribute(flac_enc_write_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)w_smem));
  flac_enc_quantise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(x, n, channels, bps, q, pcm_le_out);
  flac_enc_analyse_kernel<<<(unsigned)l.frames, ET, a_smem, stream>>>(q, ep, desc, ks, assign);
  flac_enc_write_kernel<<<(unsigned)l.frames, ET, w_smem, stream>>>(q, ep, desc, ks, assign, slots, l.slot, stat);
  flac_enc_finish_kernel<<<1, FIN_THREADS, 0, stream>>>(stat, l.frames, offsets, sum_dev);
  flac_enc_gather_kernel<<<(unsigned)l.frames, 256, 0, stream>>>(slots, l.slot, stat, offsets, frames_out, (long long)out_capacity);
  AR_CUDA_OK(cudaGetLastError());
  Summary sum;
  AR_CUDA_OK(cudaMemcpyAsync(&sum, sum_dev, sizeof(sum), cudaMemcpyDeviceToHost, stream));
  AR_CUDA_OK(cudaStreamSynchronize(stream));
  if (sum.bad_frame != LLONG_MAX) {
    char buf[200];
    std::snprintf(buf, sizeof(buf), "flac_encode: internal: frame %lld wrote %lld bits, sized %lld%s", sum.bad_frame, sum.wrote,
                  sum.sized, sum.status == ST_OVERFLOW ? " (overran its slot)" : "");
    AR_CHECK(false, AR_ERR_INVALID, buf);
  }
  *frame_bytes_total = sum.total;
  *min_frame = sum.min_bytes;
  *max_frame = sum.max_bytes;
  return AR_OK;
}

}  // namespace ar
