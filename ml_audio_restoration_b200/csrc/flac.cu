// FLAC decoder on the GPU (RFC 9639): the `sf.read` of a .flac file (src/utils/audio_processing.py:24) for the front end
// of load_audio.  Input: the bytes of the frame section of one stream (everything after the metadata blocks) and the
// STREAMINFO fields; output: planar fp32 [channels][n], x / 2^(bps-1) (soundfile's float32 read; exact for bps <= 24,
// __int2float_rn then the scale for 32-bit, as ar_pcm_to_float does).
//
// FLAC frames are independent units (sync code, header, CRC-8, subframes, CRC-16), but a sync code can also occur inside
// frame data.  The decoder:
//   1. index   : one thread per byte offset finds `FF F8|F9`, parses the header and keeps candidates whose CRC-8 is valid
//                and whose fields agree with STREAMINFO; per-block counts, one exclusive scan and a compaction pass give the
//                candidates in byte order (prefix sums, no atomics: deterministic).
//   2. walk    : one thread per candidate walks its subframes (the bitstream has no length fields, so this is serial within
//                a frame), checks the CRC-16 and records the frame's end offset and status.
//   3. chain   : on the host, from one copy of the candidate table: the true frames are the chain that starts at byte 0,
//                each next frame beginning where the previous one ends.  A break names the frame index and byte offset.
//   4. decode  : one thread per chained frame decodes again -- Rice residuals with a 64-bit bit window and __clzll for the
//                unary part, FIXED / LPC recurrence (32-bit accumulation when depth + precision + ceil(log2 order) <= 32,
//                else 64-bit, always 64-bit on the 33-bit side channel of 32-bit streams), wasted bits, stereo
//                decorrelation -- and writes the scaled samples straight into y at the frame's first sample.
// A thread per frame rather than a warp: the walk is serial anyway, and the thousands of frames of a file, in blocks of 16
// threads, spread over every SM with no idle lanes.  Every read is bounds-checked against nbytes; a malformed stream returns AR_ERR_INVALID, never faults.
#include <algorithm>
#include <cstdio>
#include <string>
#include <vector>

#include "ar_common.cuh"
#include "flac_common.cuh"

namespace ar {

namespace {

enum FlacStatus {
  FL_OK = 0, FL_NO_SYNC, FL_RESERVED_BLOCK_SIZE, FL_RESERVED_RATE, FL_RESERVED_CHANNELS, FL_RESERVED_BPS, FL_RESERVED_BIT,
  FL_BAD_NUMBER, FL_CRC8, FL_MISMATCH, FL_TRUNCATED, FL_SUBFRAME_PAD, FL_SUBFRAME_TYPE, FL_WASTED_BITS, FL_ORDER,
  FL_LPC_PRECISION, FL_LPC_SHIFT, FL_RESIDUAL_METHOD, FL_PARTITION, FL_RICE_RANGE, FL_CRC16, FL_N_STATUS
};

const char* const kStatusText[FL_N_STATUS] = {
  "ok", "no frame sync code", "reserved block-size code", "invalid sample-rate code", "reserved channel assignment",
  "reserved bit-depth code", "reserved header bit set", "invalid coded frame/sample number", "CRC-8 mismatch",
  "header disagrees with STREAMINFO (a change of block size bound, sample rate, bit depth or channel count)",
  "frame runs past the end of the data", "subframe padding bit set", "reserved subframe type", "invalid wasted-bits count",
  "predictor order larger than the partition", "invalid LPC precision", "negative LPC shift", "reserved residual coding method",
  "block size not divisible by the partition count", "Rice residual outside the 32-bit range", "CRC-16 mismatch"};

constexpr int HEADER_MAX = 16;     // sync 2 + codes 2 + coded number <= 7 + block size <= 2 + rate <= 2 + CRC-8 1
constexpr int FT = 16;             // threads per block of the walk / decode kernels: small, so that the ~2000 frames
                                   // of a 3-minute side spread over the SMs instead of filling a few
constexpr int INDEX_PER_THREAD = 4;
constexpr int INDEX_THREADS = 256;
constexpr int INDEX_SPAN = INDEX_PER_THREAD * INDEX_THREADS;   // byte offsets per index block

struct StreamParams {
  int channels, bps, sample_rate, max_block;
};

struct FlacHeader {
  int block_size, sample_rate, assign, channels, bps, variable, len;
  long long number;
};

struct FlacCand {        // one candidate frame (host copy of the table after the walk)
  long long off, end, number;
  int block_size;
  short status, variable;
};

struct FlacChain {       // one frame of the chain: where it starts in the data and in the output
  long long off, first;
};

// Frame header at p[0..avail): fields resolved against STREAMINFO (codes 0 = "from STREAMINFO").
__host__ __device__ inline int parse_header(const unsigned char* p, long long avail, const StreamParams& sp, FlacHeader* h) {
  const int have = avail < HEADER_MAX ? (int)avail : HEADER_MAX;
  if (have < 2 || p[0] != 0xFF || (p[1] & 0xFE) != 0xF8) return FL_NO_SYNC;
  if (have < 6) return FL_TRUNCATED;
  h->variable = p[1] & 1;
  const int bs_code = p[2] >> 4, rate_code = p[2] & 15, ch_code = p[3] >> 4, bps_code = (p[3] >> 1) & 7;
  if (bs_code == 0) return FL_RESERVED_BLOCK_SIZE;
  if (rate_code == 15) return FL_RESERVED_RATE;
  if (ch_code > 10) return FL_RESERVED_CHANNELS;
  if (bps_code == 3) return FL_RESERVED_BPS;
  if (p[3] & 1) return FL_RESERVED_BIT;
  // UTF-8-style coded number: up to 6 bytes (31 bits) for a frame number, 7 (36 bits) for a sample number
  int i = 4;
  const unsigned lead = p[i++];
  int extra;
  long long v;
  if (!(lead & 0x80)) { extra = 0; v = lead; }
  else if ((lead & 0xE0) == 0xC0) { extra = 1; v = lead & 0x1F; }
  else if ((lead & 0xF0) == 0xE0) { extra = 2; v = lead & 0x0F; }
  else if ((lead & 0xF8) == 0xF0) { extra = 3; v = lead & 0x07; }
  else if ((lead & 0xFC) == 0xF8) { extra = 4; v = lead & 0x03; }
  else if ((lead & 0xFE) == 0xFC) { extra = 5; v = lead & 0x01; }
  else if (lead == 0xFE && h->variable) { extra = 6; v = 0; }
  else return FL_BAD_NUMBER;
  if (i + extra > have) return FL_TRUNCATED;
  for (int k = 0; k < extra; ++k) {
    const unsigned c = p[i++];
    if ((c & 0xC0) != 0x80) return FL_BAD_NUMBER;
    v = (v << 6) | (c & 0x3F);
  }
  h->number = v;
  int bs;
  if (bs_code == 1) bs = 192;
  else if (bs_code <= 5) bs = 576 << (bs_code - 2);
  else if (bs_code == 6) { if (i + 1 > have) return FL_TRUNCATED; bs = p[i] + 1; i += 1; }
  else if (bs_code == 7) { if (i + 2 > have) return FL_TRUNCATED; bs = ((p[i] << 8) | p[i + 1]) + 1; i += 2; }
  else bs = 256 << (bs_code - 8);
  if (bs > 65535) return FL_RESERVED_BLOCK_SIZE;
  int rate;
  switch (rate_code) {
    case 0: rate = sp.sample_rate; break;
    case 1: rate = 88200; break;
    case 2: rate = 176400; break;
    case 3: rate = 192000; break;
    case 4: rate = 8000; break;
    case 5: rate = 16000; break;
    case 6: rate = 22050; break;
    case 7: rate = 24000; break;
    case 8: rate = 32000; break;
    case 9: rate = 44100; break;
    case 10: rate = 48000; break;
    case 11: rate = 96000; break;
    case 12: if (i + 1 > have) return FL_TRUNCATED; rate = p[i] * 1000; i += 1; break;
    case 13: if (i + 2 > have) return FL_TRUNCATED; rate = (p[i] << 8) | p[i + 1]; i += 2; break;
    default: if (i + 2 > have) return FL_TRUNCATED; rate = ((p[i] << 8) | p[i + 1]) * 10; i += 2; break;
  }
  if (i + 1 > have) return FL_TRUNCATED;
  if (crc8_bytes(p, i) != p[i]) return FL_CRC8;
  h->len = i + 1;
  h->block_size = bs;
  h->sample_rate = rate;
  h->assign = ch_code;
  h->channels = ch_code < 8 ? ch_code + 1 : 2;
  switch (bps_code) {
    case 0: h->bps = sp.bps; break;
    case 1: h->bps = 8; break;
    case 2: h->bps = 12; break;
    case 4: h->bps = 16; break;
    case 5: h->bps = 20; break;
    case 6: h->bps = 24; break;
    default: h->bps = 32; break;
  }
  if (h->channels != sp.channels || h->bps != sp.bps || h->sample_rate != sp.sample_rate || bs > sp.max_block)
    return FL_MISMATCH;
  return FL_OK;
}

// MSB-first reader with a left-aligned 64-bit window and the next 32-bit word already in flight (a frame is walked by one
// thread, so the load latency is what bounds it); loads past `end` read zeros and are caught by overrun().
struct BitReader {
  const unsigned char* __restrict__ p;
  long long byte, end;           // bytes [.., byte) have entered `win`; bytes [byte, byte + 4) are in `nxt`
  unsigned long long win;
  unsigned nxt;
  int cnt;

  __device__ __forceinline__ unsigned word(long long at) const {
    if (at + 4 <= end)
      return ((unsigned)__ldg(p + at) << 24) | ((unsigned)__ldg(p + at + 1) << 16) | ((unsigned)__ldg(p + at + 2) << 8) |
             (unsigned)__ldg(p + at + 3);
    unsigned w = 0;
    for (int k = 0; k < 4; ++k) w = (w << 8) | (at + k < end ? (unsigned)__ldg(p + at + k) : 0u);
    return w;
  }
  __device__ void init(const unsigned char* data, long long start, long long end_) {
    p = data; byte = start; end = end_; win = 0; cnt = 0;
    nxt = word(start);
  }
  __device__ __forceinline__ void refill() {                                        // afterwards cnt >= 32
    if (cnt > 32) return;
    win |= (unsigned long long)nxt << (32 - cnt);
    byte += 4;
    cnt += 32;
    nxt = word(byte);
  }
  __device__ __forceinline__ long long pos() const { return (byte << 3) - cnt; }        // bits consumed
  __device__ __forceinline__ bool overrun() const { return pos() > (end << 3); }
  __device__ __forceinline__ unsigned bits(int n) {                                     // 0 <= n <= 32
    if (n == 0) return 0u;
    refill();
    const unsigned v = (unsigned)(win >> (64 - n));
    win <<= n;
    cnt -= n;
    return v;
  }
  __device__ __forceinline__ long long sbits(int n) {                                   // signed, 0 <= n <= 33
    if (n == 0) return 0;
    unsigned long long u = n > 32 ? ((unsigned long long)bits(n - 32) << 32) | bits(32) : bits(n);
    return (long long)(u << (64 - n)) >> (64 - n);
  }
  // zeros before the next 1 bit (consumed); stops early (returning > limit) past `limit` zeros or the end of the data
  __device__ __forceinline__ unsigned long long unary(unsigned long long limit) {
    unsigned long long q = 0;
    for (;;) {
      refill();
      if (win != 0) break;
      q += cnt;
      win = 0;
      cnt = 0;
      if (q > limit || overrun()) return limit + 1;
    }
    const int z = __clzll((long long)win);
    q += z;
    win <<= z + 1;
    cnt -= z + 1;
    return q;
  }
  __device__ __forceinline__ void align() { const int r = cnt & 7; win <<= r; cnt -= r; }
};

__device__ __forceinline__ int ceil_log2(int v) { return v <= 1 ? 0 : 32 - __clz(v - 1); }

// Residual partitions of one subframe (method, partition order, Rice / escape codes); `emit(i, r)` receives residual r of
// sample i in order, for i in [order, bs).
template <typename Emit>
__device__ __forceinline__ int read_residual(BitReader& br, int bs, int order, Emit&& emit) {
  const int method = (int)br.bits(2);
  if (method > 1) return FL_RESIDUAL_METHOD;
  const int pbits = method == 0 ? 4 : 5, escape = (1 << pbits) - 1;
  const int porder = (int)br.bits(4);
  const int parts = 1 << porder;
  if ((bs & (parts - 1)) != 0) return FL_PARTITION;
  const int psize = bs >> porder;
  if (psize < order) return FL_ORDER;
  int i = order;
  for (int part = 0; part < parts; ++part) {
    const int count = part == 0 ? psize - order : psize;
    const int k = (int)br.bits(pbits);
    if (k == escape) {
      const int w = (int)br.bits(5);
      for (int j = 0; j < count; ++j, ++i) emit(i, (long long)br.sbits(w));
    } else {
      const unsigned long long limit = 0xFFFFFFFFull >> k;
      for (int j = 0; j < count; ++j, ++i) {
        const unsigned long long q = br.unary(limit);
        if (q > limit) return br.overrun() ? FL_TRUNCATED : FL_RICE_RANGE;
        const unsigned long long u = (q << k) | br.bits(k);
        emit(i, (long long)(u >> 1) ^ -(long long)(u & 1));
      }
    }
    if (br.overrun()) return FL_TRUNCATED;
  }
  return FL_OK;
}

// Walk (WRITE = false: status and end offset) or decode (WRITE = true: samples into y) one frame starting at byte `off`.
// Decode-only state: s_coef / s_hist are this thread's LPC coefficients and a 32-sample history ring in shared memory
// (thread-interleaved, stride FT).
template <bool WRITE>
__device__ int flac_frame(const unsigned char* __restrict__ data, long long nbytes, long long off, const StreamParams& sp,
                          float* y, long long n, long long first, int* s_coef, long long* s_hist, float scale,
                          const unsigned short* crc_tab, FlacCand* __restrict__ cand) {
  FlacHeader h;
  int st = parse_header(data + off, nbytes - off, sp, &h);
  if (st != FL_OK) return st;
  BitReader br;
  br.init(data, off + h.len, nbytes);
  const int bs = h.block_size;
  for (int ch = 0; ch < h.channels; ++ch) {
    const bool side = (h.assign == 8 && ch == 1) || (h.assign == 9 && ch == 0) || (h.assign == 10 && ch == 1);
    const int depth = h.bps + (side ? 1 : 0);
    // where the samples of this channel go: planar rows; with stereo decorrelation channel 0 is parked in row 0 as
    // int32 bits (its true value fits, or for side/right at 32 bits its low word suffices: left = side + right mod 2^32)
    // and channel 1 combines with it
    auto out = [&](int i, long long s) {
      if (!WRITE) return;
      const long long at = first + i;
      if (h.assign < 8) {
        y[ch * n + at] = __int2float_rn((int)s) * scale;
      } else if (ch == 0) {
        y[at] = __int_as_float((int)s);
      } else {
        const long long a = __float_as_int(y[at]);
        long long l, r;
        if (h.assign == 8) { l = a; r = a - s; }
        else if (h.assign == 9) { l = (int)((unsigned)a + (unsigned)s); r = s; }
        else { const long long m = (a * 2) | (s & 1); l = (m + s) >> 1; r = (m - s) >> 1; }
        y[at] = __int2float_rn((int)l) * scale;
        y[n + at] = __int2float_rn((int)r) * scale;
      }
    };
    if (br.bits(1)) return FL_SUBFRAME_PAD;
    const int type = (int)br.bits(6);
    int wasted = 0;
    if (br.bits(1)) {
      const unsigned long long q = br.unary(32);
      if (q >= 32 || (int)q + 1 >= depth) return br.overrun() ? FL_TRUNCATED : FL_WASTED_BITS;
      wasted = (int)q + 1;
    }
    const int ed = depth - wasted;
    if (type == 0) {                                             // CONSTANT
      const long long v = br.sbits(ed) * (1LL << wasted);
      if (WRITE) for (int i = 0; i < bs; ++i) out(i, v);
    } else if (type == 1) {                                      // VERBATIM
      for (int i = 0; i < bs; ++i) {
        const long long v = br.sbits(ed);
        out(i, v * (1LL << wasted));
      }
    } else if ((type & 0x38) == 0x08 && (type & 7) <= 4) {       // FIXED, order 0..4
      const int order = type & 7;
      if (order > bs) return FL_ORDER;
      long long s1 = 0, s2 = 0, s3 = 0, s4 = 0;                 // s[i-1] .. s[i-4]
      for (int i = 0; i < order; ++i) {
        const long long v = br.sbits(ed);
        s4 = s3; s3 = s2; s2 = s1; s1 = v;
        out(i, v * (1LL << wasted));
      }
      st = read_residual(br, bs, order, [&](int i, long long r) {
        if (!WRITE) return;
        long long p;
        switch (order) {
          case 0: p = 0; break;
          case 1: p = s1; break;
          case 2: p = 2 * s1 - s2; break;
          case 3: p = 3 * (s1 - s2) + s3; break;
          default: p = 4 * (s1 + s3) - 6 * s2 - s4; break;
        }
        const long long v = r + p;
        s4 = s3; s3 = s2; s2 = s1; s1 = v;
        out(i, v * (1LL << wasted));
      });
      if (st != FL_OK) return st;
    } else if (type & 0x20) {                                    // LPC, order 1..32
      const int order = (type & 31) + 1;
      if (order > bs) return FL_ORDER;
      for (int i = 0; i < order; ++i) {
        const long long v = br.sbits(ed);
        if (WRITE) s_hist[i * FT] = v;
        out(i, v * (1LL << wasted));
      }
      const int prec = (int)br.bits(4) + 1;
      if (prec == 16) return FL_LPC_PRECISION;
      const int shift = (int)br.sbits(5);
      if (shift < 0) return FL_LPC_SHIFT;
      for (int j = 0; j < order; ++j) {
        const int c = (int)br.sbits(prec);
        if (WRITE) s_coef[j * FT] = c;
      }
      const int order4 = (order + 3) & ~3;                       // zero taps up to a multiple of 4: the loops unroll by 4
      if (WRITE) for (int j = order; j < order4; ++j) s_coef[j * FT] = 0;
      const bool wide = ed + prec + ceil_log2(order) > 32;
      st = read_residual(br, bs, order, [&](int i, long long r) {
        if (!WRITE) return;
        long long p;
        if (wide) {
          long long acc = 0;
#pragma unroll 4
          for (int j = 0; j < order4; ++j) acc += (long long)s_coef[j * FT] * s_hist[((i - 1 - j) & 31) * FT];
          p = acc >> shift;
        } else {
          int acc = 0;
#pragma unroll 4
          for (int j = 0; j < order4; ++j) acc += s_coef[j * FT] * (int)s_hist[((i - 1 - j) & 31) * FT];
          p = acc >> shift;
        }
        const long long v = r + p;
        s_hist[(i & 31) * FT] = v;
        out(i, v * (1LL << wasted));
      });
      if (st != FL_OK) return st;
    } else {
      return FL_SUBFRAME_TYPE;
    }
    if (br.overrun()) return FL_TRUNCATED;
  }
  br.align();
  const unsigned stored = br.bits(16);
  if (br.overrun()) return FL_TRUNCATED;
  const long long end = br.pos() >> 3;
  if (!WRITE) {
    unsigned c = 0;
    for (long long k = off; k < end - 2; ++k) c = ((c << 8) & 0xFFFF) ^ crc_tab[((c >> 8) ^ __ldg(data + k)) & 0xFF];
    if (c != stored) return FL_CRC16;
    cand->end = end;
    cand->number = h.number;
    cand->block_size = bs;
    cand->variable = (short)h.variable;
  }
  return FL_OK;
}

__device__ __forceinline__ bool is_frame_start(const unsigned char* __restrict__ data, long long nbytes, long long i,
                                               const StreamParams& sp) {
  if (i + 1 >= nbytes || data[i] != 0xFF || (data[i + 1] & 0xFE) != 0xF8) return false;
  FlacHeader h;
  return parse_header(data + i, nbytes - i, sp, &h) == FL_OK;
}

// index pass 1/3: valid candidate headers per block of INDEX_SPAN byte offsets
__global__ void __launch_bounds__(INDEX_THREADS) flac_count_kernel(const unsigned char* __restrict__ data, long long nbytes,
                                                                   StreamParams sp, int* __restrict__ block_count) {
  __shared__ int warp_sum[INDEX_THREADS / 32];
  const long long base = (long long)blockIdx.x * INDEX_SPAN + (long long)threadIdx.x * INDEX_PER_THREAD;
  int c = 0;
  for (int k = 0; k < INDEX_PER_THREAD; ++k) c += is_frame_start(data, nbytes, base + k, sp);
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < INDEX_THREADS / 32; ++w) t += warp_sum[w];
    block_count[blockIdx.x] = t;
  }
}

// index pass 2/3: exclusive scan of the block counts (one CTA, fixed order) and the total
__global__ void __launch_bounds__(1024) flac_scan_kernel(const int* __restrict__ block_count, long long nblk,
                                                         long long* __restrict__ block_base, long long* __restrict__ total) {
  __shared__ long long part[1024];
  const long long per = (nblk + 1023) / 1024;
  const long long lo = threadIdx.x * per, hi = min(nblk, lo + per);
  long long s = 0;
  for (long long b = lo; b < hi; ++b) s += block_count[b];
  part[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long run = 0;
    for (int t = 0; t < 1024; ++t) { const long long v = part[t]; part[t] = run; run += v; }
    *total = run;
  }
  __syncthreads();
  s = part[threadIdx.x];
  for (long long b = lo; b < hi; ++b) { block_base[b] = s; s += block_count[b]; }
}

// index pass 3/3: candidate offsets in byte order at their block's base + rank within the block
__global__ void __launch_bounds__(INDEX_THREADS) flac_compact_kernel(const unsigned char* __restrict__ data, long long nbytes,
                                                                     StreamParams sp, const long long* __restrict__ block_base,
                                                                     FlacCand* __restrict__ cand, long long cap) {
  __shared__ int warp_sum[INDEX_THREADS / 32];
  const long long base = (long long)blockIdx.x * INDEX_SPAN + (long long)threadIdx.x * INDEX_PER_THREAD;
  bool ok[INDEX_PER_THREAD];
  int c = 0;
#pragma unroll
  for (int k = 0; k < INDEX_PER_THREAD; ++k) { ok[k] = is_frame_start(data, nbytes, base + k, sp); c += ok[k]; }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = c;                                                       // inclusive warp scan
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) warp_sum[warp] = incl;
  __syncthreads();
  int before = 0;
  for (int w = 0; w < warp; ++w) before += warp_sum[w];
  long long at = block_base[blockIdx.x] + before + incl - c;
#pragma unroll
  for (int k = 0; k < INDEX_PER_THREAD; ++k) {
    if (!ok[k]) continue;
    if (at < cap) {
      FlacCand e;
      e.off = base + k; e.end = -1; e.number = -1; e.block_size = 0; e.status = FL_OK; e.variable = 0;
      cand[at] = e;
    }
    ++at;
  }
}

__global__ void __launch_bounds__(FT) flac_walk_kernel(const unsigned char* __restrict__ data, long long nbytes, StreamParams sp,
                                                       FlacCand* __restrict__ cand, long long count) {
  __shared__ unsigned short tab[256];
  crc16_table(tab);
  const long long c = (long long)blockIdx.x * FT + threadIdx.x;
  if (c >= count) return;
  cand[c].status = (short)flac_frame<false>(data, nbytes, cand[c].off, sp, nullptr, 0, 0, nullptr, nullptr, 0.f, tab, cand + c);
}

__global__ void __launch_bounds__(FT) flac_decode_kernel(const unsigned char* __restrict__ data, long long nbytes, StreamParams sp,
                                                         const FlacChain* __restrict__ chain, long long frames, float* y,
                                                         long long n, float scale) {
  __shared__ int s_coef[32 * FT];
  __shared__ long long s_hist[32 * FT];
  const long long f = (long long)blockIdx.x * FT + threadIdx.x;
  if (f >= frames) return;
  const FlacChain e = chain[f];
  flac_frame<true>(data, nbytes, e.off, sp, y, n, e.first, s_coef + threadIdx.x, s_hist + threadIdx.x, scale, nullptr, nullptr);
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

struct WsLayout {
  long long nblk, cap;
  size_t counts, bases, total, cand, chain, bytes;
};

WsLayout ws_layout(long long nbytes) {
  WsLayout l;
  l.nblk = (nbytes + INDEX_SPAN - 1) / INDEX_SPAN;
  // a frame header cannot hold 0xFF in its bytes 2..4 (rate code 15, reserved bit, invalid number lead), so two
  // candidates are at least 5 bytes apart
  l.cap = nbytes / 5 + 2;
  size_t o = 0;
  l.counts = o; o += align256(sizeof(int) * (size_t)l.nblk);
  l.bases = o;  o += align256(sizeof(long long) * (size_t)l.nblk);
  l.total = o;  o += 256;
  l.cand = o;   o += align256(sizeof(FlacCand) * (size_t)l.cap);
  l.chain = o;  o += align256(sizeof(FlacChain) * (size_t)l.cap);
  l.bytes = o;
  return l;
}

std::string frame_error(long long frame, long long off, const char* what) {
  char buf[160];
  std::snprintf(buf, sizeof(buf), "FLAC: frame %lld at byte %lld: %s", frame, off, what);
  return buf;
}

}  // namespace

int flac_workspace_bytes(long long nbytes, size_t* bytes) {
  AR_CHECK(bytes && nbytes >= 0, AR_ERR_INVALID, "flac_workspace_bytes: bad argument");
  *bytes = ws_layout(nbytes).bytes;
  return AR_OK;
}

int flac_decode(const unsigned char* data, long long nbytes, int channels, int bps, int sample_rate, int min_block,
                int max_block, long long total_samples, float* y, long long n, long long* n_out, void* ws, size_t ws_bytes,
                cudaStream_t stream) {
  AR_CHECK(n_out && nbytes >= 0 && (data || nbytes == 0) && channels >= 1 && channels <= 8 && bps >= 4 && bps <= 32 &&
               sample_rate >= 1 && min_block >= 1 && max_block >= min_block && max_block <= 65535 && total_samples >= 0 && n >= 0,
           AR_ERR_INVALID, "flac_decode: bad argument");
  const WsLayout l = ws_layout(nbytes);
  AR_CHECK(ws && ws_bytes >= l.bytes, AR_ERR_WORKSPACE, "flac_decode: workspace too small (ar_flac_workspace_bytes)");
  const StreamParams sp{channels, bps, sample_rate, max_block};
  char* w = static_cast<char*>(ws);
  int* counts = reinterpret_cast<int*>(w + l.counts);
  long long* bases = reinterpret_cast<long long*>(w + l.bases);
  long long* total = reinterpret_cast<long long*>(w + l.total);
  FlacCand* cand = reinterpret_cast<FlacCand*>(w + l.cand);
  FlacChain* chain_dev = reinterpret_cast<FlacChain*>(w + l.chain);

  long long count = 0;
  if (nbytes > 0) {
    flac_count_kernel<<<(unsigned)l.nblk, INDEX_THREADS, 0, stream>>>(data, nbytes, sp, counts);
    flac_scan_kernel<<<1, 1024, 0, stream>>>(counts, l.nblk, bases, total);
    flac_compact_kernel<<<(unsigned)l.nblk, INDEX_THREADS, 0, stream>>>(data, nbytes, sp, bases, cand, l.cap);
    AR_CUDA_OK(cudaGetLastError());
    AR_CUDA_OK(cudaMemcpyAsync(&count, total, sizeof(count), cudaMemcpyDeviceToHost, stream));
    AR_CUDA_OK(cudaStreamSynchronize(stream));
    AR_CHECK(count <= l.cap, AR_ERR_INVALID, "FLAC: candidate table overflow");
  }
  std::vector<FlacCand> tab((size_t)count);
  if (count > 0) {
    flac_walk_kernel<<<(unsigned)((count + FT - 1) / FT), FT, 0, stream>>>(data, nbytes, sp, cand, count);
    AR_CUDA_OK(cudaGetLastError());
    AR_CUDA_OK(cudaMemcpyAsync(tab.data(), cand, sizeof(FlacCand) * (size_t)count, cudaMemcpyDeviceToHost, stream));
    AR_CUDA_OK(cudaStreamSynchronize(stream));
  }

  // the chain of true frames: from byte 0, each frame starts where the previous one ends
  std::vector<FlacChain> chain;
  long long pos = 0, sample = 0;
  int variable = -1;
  while (pos < nbytes && !(total_samples > 0 && sample >= total_samples)) {
    const long long f = (long long)chain.size();
    auto it = std::lower_bound(tab.begin(), tab.end(), pos, [](const FlacCand& e, long long p) { return e.off < p; });
    if (it == tab.end() || it->off != pos) {          // no valid header here: say why
      unsigned char hb[HEADER_MAX];
      const long long have = std::min<long long>(HEADER_MAX, nbytes - pos);
      AR_CUDA_OK(cudaMemcpyAsync(hb, data + pos, (size_t)have, cudaMemcpyDeviceToHost, stream));
      AR_CUDA_OK(cudaStreamSynchronize(stream));
      FlacHeader h;
      const int st = parse_header(hb, have, sp, &h);
      AR_CHECK(false, AR_ERR_INVALID, frame_error(f, pos, kStatusText[st == FL_OK ? FL_NO_SYNC : st]));
    }
    AR_CHECK(it->status == FL_OK, AR_ERR_INVALID, frame_error(f, pos, kStatusText[it->status]));
    const int var = it->variable;
    if (variable < 0) variable = var;
    AR_CHECK(var == variable, AR_ERR_INVALID, frame_error(f, pos, "blocking strategy changes mid-stream"));
    AR_CHECK(it->number == (variable ? sample : f), AR_ERR_INVALID,
             frame_error(f, pos, variable ? "coded sample number does not follow the previous frame"
                                          : "coded frame number out of sequence"));
    chain.push_back({pos, sample});
    sample += it->block_size;
    pos = it->end;
  }
  if (total_samples > 0 && sample != total_samples) {
    char buf[160];
    std::snprintf(buf, sizeof(buf), "FLAC: the frames hold %lld samples per channel, STREAMINFO says %lld%s", sample,
                  total_samples, sample < total_samples ? " (truncated stream)" : "");
    AR_CHECK(false, AR_ERR_INVALID, buf);
  }
  *n_out = sample;
  if (y == nullptr || chain.empty()) return AR_OK;
  AR_CHECK(sample <= n, AR_ERR_INVALID, "flac_decode: output rows shorter than the decoded stream");
  AR_CUDA_OK(cudaMemcpyAsync(chain_dev, chain.data(), sizeof(FlacChain) * chain.size(), cudaMemcpyHostToDevice, stream));
  const float scale = 1.0f / (float)(1LL << (bps - 1));
  const long long frames = (long long)chain.size();
  flac_decode_kernel<<<(unsigned)((frames + FT - 1) / FT), FT, 0, stream>>>(data, nbytes, sp, chain_dev, frames, y, n, scale);
  AR_CUDA_OK(cudaGetLastError());
  return AR_OK;
}

}  // namespace ar
