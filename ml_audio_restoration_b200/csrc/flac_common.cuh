// Helpers shared by the FLAC decoder (flac.cu) and encoder (flac_encode.cu): the frame-header CRC-8 (polynomial 0x07) and
// the CRC-16 table (polynomial 0x8005) of RFC 9639, both MSB-first with initial value 0 and no final xor.
#pragma once

namespace ar {

__host__ __device__ inline unsigned crc8_bytes(const unsigned char* p, int n) {
  unsigned c = 0;
  for (int i = 0; i < n; ++i) {
    c ^= p[i];
    for (int b = 0; b < 8; ++b) c = (c & 0x80) ? ((c << 1) ^ 0x07) & 0xFF : (c << 1) & 0xFF;
  }
  return c;
}

// tab[v] = v * x^16 mod P: the byte-wise update is c = ((c << 8) & 0xFFFF) ^ tab[((c >> 8) ^ byte) & 0xFF].  Built by the
// whole CTA; ends with a barrier.
__device__ inline void crc16_table(unsigned short* tab) {
  for (int v = threadIdx.x; v < 256; v += blockDim.x) {
    unsigned c = (unsigned)v << 8;
    for (int b = 0; b < 8; ++b) c = (c & 0x8000) ? ((c << 1) ^ 0x8005) & 0xFFFF : (c << 1) & 0xFFFF;
    tab[v] = (unsigned short)c;
  }
  __syncthreads();
}

}  // namespace ar
