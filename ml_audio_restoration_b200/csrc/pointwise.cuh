// Launchers of the CUDA-core kernels (pointwise.cu, lstm.cu).
#pragma once
#include <vector>

#include "ar_common.cuh"

namespace ar {

// Weights of the CUDA-core tail kernels travel as __grid_constant__ kernel parameters (the parameter space is constant
// bank 0): every FFMA then takes its weight as a c[0][imm] operand -- no weight loads at all in the inner loops.
struct alignas(16) DenTailP {   // transient detector 32->16->8->1 (k3) + final 1x1 conv, denoiser.py:39-48
  float w0[3][32][16];   // [tap][cin][cout]
  float b0[16];
  float w1[3][16][8];
  float b1[8];
  float w2[3][8];
  float wf[32];
  float b2, bf;
};
struct alignas(16) StemP {   // Cin = 1 first conv (+ folded BN): taps x 32 weights, 32 biases
  float w[7][32];        // [tap][channel]: the channel pair (2i, 2i+1) of a tap is one 8-byte constant-bank operand of a packed FFMA2
  float b[32];
  int taps;
};
struct FinalW {          // up to two 32 -> 1 k7 heads
  float w[2][7][32];     // [head][tap][cin]
  float bias[2];
};

int launch_stem(const float* x, int B, int T, const StemP& w, const Act& out, int lrelu, cudaStream_t stream);
int launch_final_k7(const Act& in, const int* in_coff8, const FinalW& w, int nout, float* y, int B, int T, const float* x_lr,
                    cudaStream_t stream);
// tensor-core version of the k7 heads (final_umma.cu): taps along N, shifted sum in the epilogue
void pack_final_umma(const FinalW& w, int nheads, std::vector<uint16_t>& out);
int launch_final_umma(const Act& in, int in_coff8, const __half* w_packed, const FinalW& w, int nheads, float* y, int B, int T,
                      const float* x_lr, cudaStream_t stream);
// h1 != nullptr: the first detector layer already ran in the conv engine (H8, channels 0..15 of *h1)
int launch_den_tail(const Act& f, const Act* h1, const float* x, float* y, int B, int T, const DenTailP& w, cudaStream_t stream);
int launch_normalize(float* x, long long n, float target_db, float* scratch, cudaStream_t stream);
int launch_split(const float* audio, long long n, float* chunks, int first, int count, int chunk_size, int overlap,
                 cudaStream_t stream);
int launch_ola(const float* y, float* out, long long n, int n_chunks, int channels, int chunk_size, int overlap, int rate,
               cudaStream_t stream);
// max |value| over rows [0,T) of channel chunks [coff8, coff8 + nch8) of an activation tensor -> atomic max into *slot
// (float bits); dynamic-range audit
int launch_audit(const Act& a, int B, int coff8, int nch8, int T, int tblock, unsigned int* slot, cudaStream_t stream);
// the same window as plain fp32 [B][8 nch8][T] (ar_model_audit_tap)
int launch_audit_tap(const Act& a, int B, int coff8, int nch8, int T, int tblock, float* y, cudaStream_t stream);
int launch_plain_to_c4(const float* x, int B, int C, int T, const Act& out, cudaStream_t stream);
int launch_c4_to_plain(const Act& in, int B, int C, int T, float* y, cudaStream_t stream);

// xp: H8 fp16 [B][256 ch] gate pre-activations (W_ih x + b_ih + b_hh, rows i|f|g|o), whh: [256][64] device,
// h_out: H8 fp16 [B][64 ch]; state_in/out: [B][2][64] (h, c) or nullptr.
int launch_lstm(const Act& xp, const float* whh, const Act& h_out, int B, int T, const float* state_in, float* state_out,
                cudaStream_t stream);
// scan that computes its own input projection on the tensor pipe (lstm_proj.cu): x = encoder output, 128 channels
void pack_lstm_proj(const float* G, std::vector<uint16_t>& out);
int launch_lstm_proj(const Act& x, const __half* wih_packed, const float* bias, const float* whh, const Act& h_out, int B, int T,
                     const float* state_in, float* state_out, cudaStream_t stream);

}  // namespace ar
