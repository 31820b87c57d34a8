// Host side of libaudiorestore_sm100: state_dict -> folded / packed device weights, the
// workspace planner, and the three model forwards + the chain expressed as kernel sequences.
#include <atomic>
#include <cmath>
#include <cuda_fp16.h>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "ar_common.cuh"
#include "pointwise.cuh"
#include "prof.cuh"

namespace ar {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* last_error() { return g_err.c_str(); }
// Process-wide knobs read when a model is created (cross-check / tuning hooks of the C-ABI, no environment variables).
static std::atomic<int> g_engine{AR_ENGINE_UMMA};
int set_engine(int e) {
  if (e != AR_ENGINE_UMMA && e != AR_ENGINE_SIMT) { set_error("unknown conv engine"); return AR_ERR_INVALID; }
  g_engine.store(e);
  return AR_OK;
}
// Fused multi-layer launches (conv_chain.cu) for subsequently created models: 0 = layer by layer, 1 = every chain that
// fits (product default)
static std::atomic<bool> g_fuse{true};
int set_fusion(int on) {
  if (on != 0 && on != 1) { set_error("fusion must be 0 (layer by layer) or 1 (fused)"); return AR_ERR_INVALID; }
  g_fuse.store(on == 1);
  return AR_OK;
}
static std::atomic<long long*> g_chain_trace{nullptr};   // debug: device buffer the fused-chain kernels trace their pipeline into
static std::atomic<int> g_chain_trace_slot{0};           // launch k after ar_debug_chain_trace() writes slot k % 8 of [8][64*16]
int set_chain_trace(long long* dev_buf) { g_chain_trace.store(dev_buf); g_chain_trace_slot.store(0); return AR_OK; }

// ============================================================================ weight folding / packing
static uint16_t half_bits_host(float x) {  // fp32 -> fp16, round to nearest even, clamped to the finite range
  if (x > 65504.f) x = 65504.f;
  if (x < -65504.f) x = -65504.f;
  const __half h = __float2half_rn(x);
  uint16_t b;
  std::memcpy(&b, &h, 2);
  return b;
}

struct Table {
  std::map<std::string, const ar_tensor_t*> m;
  const float* get(const std::string& name, std::initializer_list<int64_t> shape) const {
    auto it = m.find(name);
    if (it == m.end()) { set_error("Missing key(s) in state_dict: \"" + name + "\""); return nullptr; }
    const ar_tensor_t* t = it->second;
    bool ok = t->ndim == (int)shape.size() && t->data != nullptr;
    int i = 0;
    for (int64_t s : shape) { if (ok && t->shape[i] != s) ok = false; ++i; }
    if (!ok) { set_error("size mismatch for " + name); return nullptr; }
    return t->data;
  }
};

// A conv expressed as the GEMM the engines run: G[tap][cin][n] (+ bias[n]).
struct Gemm {
  int Cin = 0, N = 0, taps = 1, dil = 1, pad_left = 0;
  std::vector<float> G, bias;
  void init(int cin, int n, int t, int d, int pl) {
    Cin = cin; N = n; taps = t; dil = d; pad_left = pl;
    G.assign((size_t)t * cin * n, 0.f);
    bias.assign(n, 0.f);
  }
  float& at(int tap, int cin, int n) { return G[((size_t)tap * Cin + cin) * N + n]; }
};

struct ConvLayer {  // device-resident packed layer
  int Cin, N, taps, dil, pad_left;
  size_t w_off, b_off;  // float offsets into the model blob
  double macs_per_row;  // algorithmic MACs of the reference op per input time step (structural zeros excluded)
  int n_slices;         // column slices (each slice's weights stay resident in one CTA's shared memory)
  int cta2;             // slices come in (2i, 2i+1) pairs: the two halves of a 2-CTA pair-slice
};

// Resident-weight budget per CTA (fp16 weights): leaves >= ~96 KB of the 227 KB for the activation ring.
// With the 2-CTA engine every layer of the three models fits unsliced (largest: 256x256 k3 = 192 KB / CTA).
constexpr size_t W_SLICE_BUDGET = 128 * 1024;
static int pick_slices(int Cin, int taps, int N) {
  int s = 1;
  while ((size_t)Cin * taps * (N / s) * 2 > W_SLICE_BUDGET && (N / (2 * s)) % 16 == 0) s *= 2;
  return s;
}
// Every layer with N a multiple of 32 is packed as pair-slices of two halves (one per CTA of the 2-CTA engine).
static bool want_cta2(int N) { return N >= 32 && N % 32 == 0; }

struct Blob {
  std::vector<float> host;
  // Largest |folded weight| seen and the smallest per-layer maximum: operands are stored in fp16 (finite range 65504,
  // normal range down to 6.1e-5), so a BN fold with a tiny running_var can push a layer outside it.
  float w_max = 0.f, w_min_layer_max = 1e30f;
  size_t push(const float* p, size_t n) {
    size_t off = (host.size() + 63) / 64 * 64;  // 256-byte aligned
    host.resize(off + n);
    std::memcpy(host.data() + off, p, n * sizeof(float));
    return off;
  }
  size_t push(const std::vector<float>& v) { return push(v.data(), v.size()); }
  size_t push_half(const std::vector<uint16_t>& h) {   // a packed fp16 operand, zero-padded to whole floats
    std::vector<float> raw((h.size() + 1) / 2);
    std::memcpy(raw.data(), h.data(), h.size() * 2);
    return push(raw);
  }
  ConvLayer push_gemm(Gemm& g) {  // fp16 [n_slices][Cin/16][taps][2][Ns][8]
    const bool cta2 = want_cta2(g.N);
    // per-CTA slices: for the 2-CTA engine split every pair-slice once more (the budget applies per CTA)
    int ns = pick_slices(g.Cin, g.taps, g.N);
    if (cta2 && ns == 1) ns = 2;
    const int Ns = g.N / ns, KB = g.Cin / 16;
    std::vector<uint16_t> w((size_t)g.Cin * g.taps * g.N);
    for (int sl = 0; sl < ns; ++sl)
      for (int kb = 0; kb < KB; ++kb)
        for (int t = 0; t < g.taps; ++t)
          for (int h = 0; h < 2; ++h)
            for (int n = 0; n < Ns; ++n)
              for (int j = 0; j < 8; ++j)
                w[(((((size_t)sl * KB + kb) * g.taps + t) * 2 + h) * Ns + n) * 8 + j] =
                    half_bits_host(g.at(t, kb * 16 + h * 8 + j, sl * Ns + n));
    ConvLayer L{g.Cin, g.N, g.taps, g.dil, g.pad_left, 0, 0, 0.0, ns, cta2 ? 1 : 0};
    float lmax = 0.f;
    for (float v : g.G) {
      L.macs_per_row += (v != 0.f) ? 1.0 : 0.0;  // == Cin*N*taps except the 2-phase ConvT
      const float av = std::fabs(v);
      if (!(av <= lmax)) lmax = av;               // also catches NaN
    }
    if (!(lmax <= w_max)) w_max = lmax;
    if (lmax < w_min_layer_max) w_min_layer_max = lmax;
    L.w_off = push_half(w);
    L.b_off = push(g.bias);
    return L;
  }
};

// BN(eval) fold: s = gamma / sqrt(var + eps); W' = W*s; b' = (b - mean)*s + beta  (App. B.4)
struct Fold { std::vector<float> s, b; };
static bool fold_bn(const Table& t, const std::string& conv, const std::string& bn, int cout, Fold& f) {
  const float* b = t.get(conv + ".bias", {cout});
  if (!b) return false;
  f.s.assign(cout, 1.f);
  f.b.assign(b, b + cout);
  if (bn.empty()) return true;
  const float* g = t.get(bn + ".weight", {cout});
  const float* be = t.get(bn + ".bias", {cout});
  const float* mu = t.get(bn + ".running_mean", {cout});
  const float* var = t.get(bn + ".running_var", {cout});
  if (!g || !be || !mu || !var) return false;
  float eps = 1e-5f;                                   // nn.BatchNorm1d default; "<bn>.eps" ([1]) overrides it
  auto it = t.m.find(bn + ".eps");
  if (it != t.m.end() && it->second->data != nullptr) eps = it->second->data[0];
  for (int o = 0; o < cout; ++o) {
    const float s = g[o] / std::sqrt(var[o] + eps);
    f.s[o] = s;
    f.b[o] = (b[o] - mu[o]) * s + be[o];
  }
  return true;
}

// nn.Conv1d(cin, cout, k, padding=dil*(k-1)/2, dilation=dil) [+ BN] into columns [n_off, n_off+cout) of g.
static bool add_conv(const Table& t, const std::string& conv, const std::string& bn, int cin, int cout, int k, Gemm& g, int n_off = 0) {
  const float* W = t.get(conv + ".weight", {cout, cin, k});
  Fold f;
  if (!W || !fold_bn(t, conv, bn, cout, f)) return false;
  for (int o = 0; o < cout; ++o) {
    for (int c = 0; c < cin; ++c)
      for (int j = 0; j < k; ++j) g.at(j, c, n_off + o) = W[((size_t)o * cin + c) * k + j] * f.s[o];
    g.bias[n_off + o] = f.b[o];
  }
  return true;
}

static bool make_conv(const Table& t, Blob& blob, const std::string& conv, const std::string& bn, int cin, int cout, int k, int dil,
                      ConvLayer& out) {
  Gemm g;
  g.init(cin, cout, k, dil, dil * (k - 1) / 2);
  if (!add_conv(t, conv, bn, cin, cout, k, g)) return false;
  out = blob.push_gemm(g);
  return true;
}

// ============================================================================ model objects

struct Model {
  int kind = -1, device = 0, engine = AR_ENGINE_UMMA;
  bool fuse = true;   // fused conv chains (tcgen05 engine, 2-CTA packing) wherever the chain kernel takes the layers
  float* blob = nullptr;
  std::map<std::string, ConvLayer> conv;
  StemP stem{};          // Cin = 1 stem: kernel-parameter weights
  // CUDA-core tails: weights live on the host and travel as kernel parameters (constant bank)
  DenTailP den_tail{};   // denoiser: transient detector + final 1x1
  FinalW fin{};          // final k7 convs (sr: 1 head, stereo: 2)
  size_t fin_umma_off = 0;   // the same heads packed as a tap-along-N tensor-core operand (final_umma.cu)
  int fin_heads = 0;
  size_t whh_off = 0;
  size_t wih_umma_off = 0;   // W_ih^T packed for the scan kernel that computes its own input projection (lstm_proj.cu)
  // dynamic-range audit (ar_model_audit_*): while on, forwards run layer by layer and fold max |activation| of every
  // fp16 tensor they write into audit_dev[slot]; names are recorded in launch order.  Not re-entrant.
  bool audit = false;
  unsigned int* audit_dev = nullptr;
  std::vector<std::string> audit_names;
  struct Tap { float* y; long long cap; };
  std::map<std::string, Tap> audit_taps;   // ar_model_audit_tap: audited tensors also copied out as plain fp32
  ~Model() { if (blob) cudaFree(blob); if (audit_dev) cudaFree(audit_dev); }
};
constexpr int AUDIT_SLOTS = AR_AUDIT_MAX_LAYERS;

static bool stem_pack(const Table& t, const std::string& conv, const std::string& bn, int k, StemP& s) {
  const float* W = t.get(conv + ".weight", {32, 1, k});
  Fold f;
  if (!W || !fold_bn(t, conv, bn, 32, f)) return false;
  std::memset(&s, 0, sizeof(s));
  for (int o = 0; o < 32; ++o) {
    for (int j = 0; j < k; ++j) s.w[j][o] = W[o * k + j] * f.s[o];
    s.b[o] = f.b[o];
  }
  s.taps = k;
  return true;
}

static bool build_denoiser(const Table& t, Blob& blob, Model& m) {
  const int F[3] = {32, 64, 128};
  if (!stem_pack(t, "encoder.0.0", "encoder.0.1", 3, m.stem)) return false;
  if (!make_conv(t, blob, "encoder.0.3", "encoder.0.4", 32, 32, 3, 1, m.conv["enc0b"])) return false;
  if (!make_conv(t, blob, "encoder.1.0", "encoder.1.1", 32, 64, 3, 1, m.conv["enc1a"])) return false;
  if (!make_conv(t, blob, "encoder.1.3", "encoder.1.4", 64, 64, 3, 1, m.conv["enc1b"])) return false;
  if (!make_conv(t, blob, "encoder.2.0", "encoder.2.1", 64, 128, 3, 1, m.conv["enc2a"])) return false;
  if (!make_conv(t, blob, "encoder.2.3", "encoder.2.4", 128, 128, 3, 1, m.conv["enc2b"])) return false;
  if (!make_conv(t, blob, "bottleneck.0", "bottleneck.1", 128, 256, 3, 1, m.conv["bot_a"])) return false;
  if (!make_conv(t, blob, "bottleneck.3", "bottleneck.4", 256, 256, 3, 1, m.conv["bot_b"])) return false;
  for (int i = 0; i < 3; ++i) {
    const int f = F[2 - i];
    const std::string up = "decoder." + std::to_string(2 * i), blk = "decoder." + std::to_string(2 * i + 1);
    // ConvTranspose1d(2f, f, k=2, s=2): y[2t+j] = W[:,:,j]^T x[t] + b  (App. B.1) -> N = 2f, columns [j*f + o]
    const float* W = t.get(up + ".weight", {2 * f, f, 2});
    const float* b = t.get(up + ".bias", {f});
    if (!W || !b) return false;
    Gemm g;
    g.init(2 * f, 2 * f, 1, 1, 0);
    for (int c = 0; c < 2 * f; ++c)
      for (int o = 0; o < f; ++o)
        for (int j = 0; j < 2; ++j) g.at(0, c, j * f + o) = W[((size_t)c * f + o) * 2 + j];
    for (int o = 0; o < f; ++o) g.bias[o] = g.bias[f + o] = b[o];
    m.conv["up" + std::to_string(i)] = blob.push_gemm(g);
    if (!make_conv(t, blob, blk + ".0", blk + ".1", 2 * f, f, 3, 1, m.conv["dec" + std::to_string(i) + "a"])) return false;
    if (!make_conv(t, blob, blk + ".3", blk + ".4", f, f, 3, 1, m.conv["dec" + std::to_string(i) + "b"])) return false;
  }
  // transient detector + final conv (CUDA-core tail kernel)
  const float* W0 = t.get("transient_detector.0.weight", {16, 32, 3});
  const float* B0 = t.get("transient_detector.0.bias", {16});
  const float* W1 = t.get("transient_detector.2.weight", {8, 16, 3});
  const float* B1 = t.get("transient_detector.2.bias", {8});
  const float* W2 = t.get("transient_detector.4.weight", {1, 8, 3});
  const float* B2 = t.get("transient_detector.4.bias", {1});
  const float* WF = t.get("final_conv.weight", {1, 32, 1});
  const float* BF = t.get("final_conv.bias", {1});
  if (!W0 || !B0 || !W1 || !B1 || !W2 || !B2 || !WF || !BF) return false;
  DenTailP& P = m.den_tail;
  for (int j = 0; j < 3; ++j) {
    for (int c = 0; c < 32; ++c)
      for (int o = 0; o < 16; ++o) P.w0[j][c][o] = W0[(o * 32 + c) * 3 + j];
    for (int c = 0; c < 16; ++c)
      for (int o = 0; o < 8; ++o) P.w1[j][c][o] = W1[(o * 16 + c) * 3 + j];
    for (int c = 0; c < 8; ++c) P.w2[j][c] = W2[c * 3 + j];
  }
  for (int o = 0; o < 16; ++o) P.b0[o] = B0[o];
  for (int o = 0; o < 8; ++o) P.b1[o] = B1[o];
  for (int c = 0; c < 32; ++c) P.wf[c] = WF[c];
  P.b2 = B2[0];
  P.bf = BF[0];
  // the first detector layer (32 -> 16 k3 + LeakyReLU, denoiser.py:40-41) as a conv-engine layer: padded to 32 output
  // columns (zero weights / bias) so that it runs in the 2-CTA engine with tile groups like the other 32-channel layers
  Gemm g;
  g.init(32, 32, 3, 1, 1);
  if (!add_conv(t, "transient_detector.0", "", 32, 16, 3, g, 0)) return false;
  m.conv["td0"] = blob.push_gemm(g);
  return true;
}

static bool build_sr(const Table& t, Blob& blob, Model& m) {
  if (!stem_pack(t, "initial.0", "", 7, m.stem)) return false;
  for (int i = 0; i < 4; ++i) {
    const std::string p = "residual_blocks." + std::to_string(i);
    if (!make_conv(t, blob, p + ".conv1", p + ".bn1", 32, 32, 3, 1, m.conv["rb" + std::to_string(i) + "a"])) return false;
    if (!make_conv(t, blob, p + ".conv2", p + ".bn2", 32, 32, 3, 1, m.conv["rb" + std::to_string(i) + "b"])) return false;
  }
  if (!make_conv(t, blob, "middle.0", "middle.1", 32, 32, 3, 1, m.conv["middle"])) return false;
  // ConvTranspose1d(32,32,k=4,s=2,p=1) as a 3-tap, 2-phase conv (App. B.2):
  //   y[2t]   = W[..,1]^T x[t] + W[..,3]^T x[t-1]      -> columns [0,32)
  //   y[2t+1] = W[..,2]^T x[t] + W[..,0]^T x[t+1]      -> columns [32,64)
  const float* W = t.get("upsample_blocks.0.0.weight", {32, 32, 4});
  const float* b = t.get("upsample_blocks.0.0.bias", {32});
  if (!W || !b) return false;
  Gemm g;
  g.init(32, 64, 3, 1, 1);
  for (int c = 0; c < 32; ++c)
    for (int o = 0; o < 32; ++o) {
      const float* w4 = W + ((size_t)c * 32 + o) * 4;
      g.at(0, c, o) = w4[3];
      g.at(1, c, o) = w4[1];
      g.at(1, c, 32 + o) = w4[2];
      g.at(2, c, 32 + o) = w4[0];
    }
  for (int o = 0; o < 32; ++o) g.bias[o] = g.bias[32 + o] = b[o];
  m.conv["up"] = blob.push_gemm(g);
  if (!make_conv(t, blob, "hf_emphasis.0", "", 32, 32, 5, 1, m.conv["hf"])) return false;
  const float* WR = t.get("reconstruction.weight", {1, 32, 7});
  const float* BR = t.get("reconstruction.bias", {1});
  if (!WR || !BR) return false;
  // The head's weights are rounded to fp16 for BOTH ways it runs (fused behind hf_emphasis on the tensor core; CUDA-core
  // kernel layer by layer), so the two paths compute from the same operands
  auto r16 = [](float v) { const uint16_t b = half_bits_host(v); __half h; std::memcpy(&h, &b, 2); return __half2float(h); };
  Gemm gh;
  gh.init(32, 32, 7, 1, 3);
  for (int c = 0; c < 32; ++c)
    for (int j = 0; j < 7; ++j) {
      m.fin.w[0][j][c] = r16(WR[c * 7 + j]);
      gh.at(j, c, 0) = WR[c * 7 + j];
    }
  gh.bias[0] = BR[0];
  m.conv["head"] = blob.push_gemm(gh);
  m.fin.bias[0] = BR[0];
  m.fin_heads = 1;
  std::vector<uint16_t> pk;
  pack_final_umma(m.fin, 1, pk);
  m.fin_umma_off = blob.push_half(pk);
  return true;
}

static bool build_stereo(const Table& t, Blob& blob, Model& m) {
  if (!stem_pack(t, "encoder.0.0", "encoder.0.1", 7, m.stem)) return false;
  const int dims[4][2] = {{32, 64}, {64, 128}, {128, 128}, {128, 128}};
  for (int i = 0; i < 4; ++i) {
    const std::string p = "encoder." + std::to_string(i + 1);
    if (!make_conv(t, blob, p + ".0", p + ".1", dims[i][0], dims[i][1], 3, 1 << i, m.conv["enc" + std::to_string(i + 1) + "a"])) return false;
    if (!make_conv(t, blob, p + ".3", p + ".4", dims[i][1], dims[i][1], 1, 1, m.conv["enc" + std::to_string(i + 1) + "b"])) return false;
  }
  // LSTM input projection as a k=1 conv 128 -> 256 with bias b_ih + b_hh (App. B.5)
  const float* Wih = t.get("lstm.weight_ih_l0", {256, 128});
  const float* Whh = t.get("lstm.weight_hh_l0", {256, 64});
  const float* bih = t.get("lstm.bias_ih_l0", {256});
  const float* bhh = t.get("lstm.bias_hh_l0", {256});
  if (!Wih || !Whh || !bih || !bhh) return false;
  // Output channels are permuted to [unit][gate] (gate order i,f,g,o) so that the four gate pre-activations a
  // recurrence thread needs are 8 contiguous bytes of the H8 tensor.
  // Rows are pre-scaled so that the recurrence kernels' gate functions are bare ex2's (lstm.cu, lstm_cell): log2(e) for the
  // i, f, o gates, 2 log2(e) for the cell candidate g -- applied to W_ih, both biases and W_hh alike.
  const float L2E = 1.4426950408889634f;
  const float gate_scale[4] = {L2E, L2E, 2.0f * L2E, L2E};
  Gemm g;
  g.init(128, 256, 1, 1, 0);
  for (int o = 0; o < 256; ++o) {
    const int op = (o % 64) * 4 + o / 64;
    const float sc = gate_scale[o / 64];
    for (int c = 0; c < 128; ++c) g.at(0, c, op) = Wih[o * 128 + c] * sc;
    g.bias[op] = (bih[o] + bhh[o]) * sc;
  }
  m.conv["xproj"] = blob.push_gemm(g);
  std::vector<uint16_t> pk;
  pack_lstm_proj(g.G.data(), pk);
  m.wih_umma_off = blob.push_half(pk);
  {
    std::vector<float> whh_s(256 * 64);
    for (int o = 0; o < 256; ++o)
      for (int k = 0; k < 64; ++k) whh_s[o * 64 + k] = Whh[o * 64 + k] * gate_scale[o / 64];
    m.whh_off = blob.push(whh_s);
  }
  // decoders: first layers of L and R share their input -> one GEMM with N = 256
  Gemm d0;
  d0.init(64, 256, 7, 1, 3);
  if (!add_conv(t, "left_decoder.0", "left_decoder.1", 64, 128, 7, d0, 0)) return false;
  if (!add_conv(t, "right_decoder.0", "right_decoder.1", 64, 128, 7, d0, 128)) return false;
  m.conv["dec0"] = blob.push_gemm(d0);
  const char* sides[2] = {"left_decoder", "right_decoder"};
  for (int s = 0; s < 2; ++s) {
    const std::string p = sides[s], tag = s ? "R" : "L";
    if (!make_conv(t, blob, p + ".3", p + ".4", 128, 64, 7, 1, m.conv["dec1" + tag])) return false;
    if (!make_conv(t, blob, p + ".6", p + ".7", 64, 32, 7, 1, m.conv["dec2" + tag])) return false;
    const float* WF = t.get(p + ".9.weight", {1, 32, 7});
    const float* BF = t.get(p + ".9.bias", {1});
    if (!WF || !BF) return false;
    for (int c = 0; c < 32; ++c)
      for (int j = 0; j < 7; ++j) m.fin.w[s][j][c] = WF[c * 7 + j];
    m.fin.bias[s] = BF[0];
  }
  m.fin_heads = 2;
  pack_final_umma(m.fin, 2, pk);
  m.fin_umma_off = blob.push_half(pk);
  return true;
}

int model_create(int kind, const ar_tensor_t* tensors, int n, int device, Model** out) {
  AR_CHECK(out != nullptr && (tensors != nullptr || n == 0), AR_ERR_INVALID, "model_create: null argument");
  int ndev = 0;
  AR_CUDA_OK(cudaGetDeviceCount(&ndev));
  AR_CHECK(device >= 0 && device < ndev, AR_ERR_CUDA, "model_create: no such CUDA device (this library has no CPU fallback)");
  cudaDeviceProp prop;
  AR_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  AR_CHECK(prop.major == 10, AR_ERR_CUDA, std::string("model_create: device is sm_") + std::to_string(prop.major * 10 + prop.minor) + ", this library is built for sm_100a only");
  Table t;
  for (int i = 0; i < n; ++i) t.m[tensors[i].name] = &tensors[i];
  std::unique_ptr<Model> m(new Model);
  m->kind = kind;
  m->device = device;
  m->engine = g_engine.load();
  m->fuse = m->engine == AR_ENGINE_UMMA && g_fuse.load();
  Blob blob;
  bool ok = false;
  if (kind == AR_MODEL_DENOISER) ok = build_denoiser(t, blob, *m);
  else if (kind == AR_MODEL_SUPER_RES) ok = build_sr(t, blob, *m);
  else if (kind == AR_MODEL_STEREO) ok = build_stereo(t, blob, *m);
  else { set_error("model_create: unknown model kind"); return AR_ERR_INVALID; }
  if (!ok) return AR_ERR_WEIGHTS;
  // Dynamic-range envelope of the fp16 operand storage (INTEGRATION.md): refuse a checkpoint whose BN-folded weights do
  // not fit instead of silently clamping them.
  if (!(blob.w_max <= HALF_MAX)) {
    set_error("model_create: a BatchNorm-folded conv weight is " + std::to_string(blob.w_max) +
              " (or not finite): outside the fp16 operand range of the tensor-core path (|w| <= 65504); "
              "check running_var / weight of the checkpoint's BatchNorm layers");
    return AR_ERR_WEIGHTS;
  }
  if (blob.w_min_layer_max > 0.f && blob.w_min_layer_max < 6.2e-5f) {
    set_error("model_create: every BatchNorm-folded weight of one conv layer is below the fp16 normal range (max " +
              std::to_string(blob.w_min_layer_max) + "): the tensor-core path would lose its precision");
    return AR_ERR_WEIGHTS;
  }
  AR_CUDA_OK(cudaSetDevice(device));
  AR_CUDA_OK(cudaMalloc(&m->blob, blob.host.size() * sizeof(float)));
  AR_CUDA_OK(cudaMemcpy(m->blob, blob.host.data(), blob.host.size() * sizeof(float), cudaMemcpyHostToDevice));
  *out = m.release();
  return AR_OK;
}

// ============================================================================ workspace arena
// Two-ended first-fit arena over the caller's workspace.  The same allocation sequence runs in a dry pass (sizes only)
// to answer *_workspace_bytes and in the real pass.  A forward is a chain of producer -> consumer tensors with two or three
// alive at a time; a one-ended first-fit arena fragments on it (a freed input is never large enough for the next, larger,
// output: 608 instead of 384 channel-planes at the stereo stage's peak, 103 instead of 68 MB per 2 s chunk).  Here a new
// tensor goes into a hole if one fits, else to the shorter END (low or high) of the workspace, so consecutive tensors
// alternate sides and the peak is the largest pair alive together.  High-side offsets count down from `cap`, the dry-run
// peak, which the real pass therefore needs before it starts.
struct Arena {
  char* base = nullptr;
  size_t cap = 0, peak = 0;
  bool dry = true;
  struct Blk { size_t off, size; bool used; };
  struct Side {
    std::vector<Blk> blks;     // sorted by offset from this side's end of the workspace
    size_t extent() const {    // bytes from this end up to the last used block
      for (size_t i = blks.size(); i-- > 0;)
        if (blks[i].used) return blks[i].off + blks[i].size;
      return 0;
    }
    // extent after a first-fit placement of `bytes` (not committed)
    size_t extent_with(size_t bytes) const {
      const size_t e = extent();
      for (const Blk& b : blks)
        if (!b.used && b.size >= bytes && b.off + b.size <= e) return e;   // fits into a hole below the extent
      size_t off = 0;
      for (size_t i = blks.size(); i-- > 0;)
        if (blks[i].used) { off = blks[i].off + blks[i].size; break; }
      return off + bytes;
    }
    size_t alloc(size_t bytes) {
      const size_t e = extent();
      for (size_t i = 0; i < blks.size(); ++i)
        if (!blks[i].used && blks[i].size >= bytes && blks[i].off + blks[i].size <= e) {
          if (blks[i].size > bytes) {
            Blk rest{blks[i].off + bytes, blks[i].size - bytes, false};
            blks[i].size = bytes;
            blks.insert(blks.begin() + i + 1, rest);
          }
          blks[i].used = true;
          return blks[i].off;
        }
      while (!blks.empty() && !blks.back().used) blks.pop_back();   // free tail: re-grow from the last used block
      const size_t off = blks.empty() ? 0 : blks.back().off + blks.back().size;
      blks.push_back({off, bytes, true});
      return off;
    }
    bool release(size_t off) {
      for (size_t i = 0; i < blks.size(); ++i)
        if (blks[i].off == off && blks[i].used) {
          blks[i].used = false;
          if (i + 1 < blks.size() && !blks[i + 1].used) { blks[i].size += blks[i + 1].size; blks.erase(blks.begin() + i + 1); }
          if (i > 0 && !blks[i - 1].used) { blks[i - 1].size += blks[i].size; blks.erase(blks.begin() + i); }
          return true;
        }
      return false;
    }
  };
  Side lo, hi;
  // returns the byte offset from `base`
  size_t alloc(size_t bytes) {
    bytes = (bytes + 255) / 256 * 256;
    // a hole below a side's extent costs nothing; otherwise grow the SHORTER side: the tensor just produced sits on the other
    // one and the one before it is about to be released, so consecutive tensors alternate ends
    const bool fits_lo = lo.extent_with(bytes) == lo.extent(), fits_hi = hi.extent_with(bytes) == hi.extent();
    const bool low = fits_lo ? true : (fits_hi ? false : lo.extent() <= hi.extent());
    const size_t off = low ? lo.alloc(bytes) : hi.alloc(bytes);
    const size_t total = lo.extent() + hi.extent();
    if (total > peak) peak = total;
    return low ? off : cap - off - bytes;          // dry pass: cap == 0, the value is not used as an address
  }
  void release_off(size_t off_from_base) {
    if (lo.release(off_from_base)) return;
    for (const Blk& b : hi.blks)            // high side: block offsets count down from `cap`
      if (b.used && cap - b.off - b.size == off_from_base) { hi.release(b.off); return; }
  }
  Act act(int B, int C, int T) {
    Act a;
    a.C = C; a.T = T; a.Tp = padded_rows(T);
    a.bs = (long long)C * a.Tp;
    const size_t off = alloc((size_t)B * a.bs * 2);
    a.base = base + off;
    return a;
  }
  void release(const Act& a) { release_off((size_t)(reinterpret_cast<char*>(a.base) - base)); }
  float* plain(size_t floats) { return reinterpret_cast<float*>(base + alloc(floats * sizeof(float))); }
  void release_plain(const float* p) { release_off((size_t)(reinterpret_cast<const char*>(p) - base)); }
};

struct Ctx {
  Arena ar;
  cudaStream_t stream = nullptr;
  int B = 0;
  const Model* m = nullptr;
};

struct ConvOpt {
  int in_coff8 = 0, out_coff8 = 0;   // channel offsets in units of 8 channels
  int mode = MODE_SAME;
  int lrelu = 1;
  int out_tblock = 0;
  const Act* pool = nullptr;
  const Act* res = nullptr;
  int Tout = -1;
  float* head_y = nullptr;          // fused output head (run_chain only): plain fp32 output and the low-rate interpolation source
  const float* head_xlr = nullptr;
};

// Dynamic-range audit hook: fold max |value| of the channel window a layer just wrote into the model's audit slot `name`.
static int audit_act(Ctx& c, const std::string& name, const Act& a, int coff8, int nch8, int T, int tblock = 0) {
  if (c.ar.dry || !c.m->audit) return AR_OK;
  Model* m = const_cast<Model*>(c.m);
  size_t slot = 0;
  while (slot < m->audit_names.size() && m->audit_names[slot] != name) ++slot;
  if (slot == m->audit_names.size()) {
    AR_CHECK(slot < (size_t)AUDIT_SLOTS, AR_ERR_INVALID, "internal: too many audited layers");
    m->audit_names.push_back(name);
  }
  auto tap = m->audit_taps.find(name);
  if (tap != m->audit_taps.end()) {
    const long long n = (long long)c.B * nch8 * 8 * T;
    AR_CHECK(n <= tap->second.cap, AR_ERR_INVALID,
             "audit tap " + name + ": window of " + std::to_string(n) + " floats exceeds the buffer (" + std::to_string(tap->second.cap) + ")");
    AR_TRY(launch_audit_tap(a, c.B, coff8, nch8, T, tblock, tap->second.y, c.stream));
  }
  return launch_audit(a, c.B, coff8, nch8, T, tblock, m->audit_dev + slot, c.stream);
}

// Launch parameters of layer `L` (offsets into the weight blob `blob`) from `in` to `out`; `stride` = output rows per tile.
static ConvParams conv_params(const ConvLayer& L, const float* blob, const Act& in, const Act& out, const ConvOpt& o, int B, int stride) {
  ConvParams p;
  std::memset(&p, 0, sizeof(p));
  p.in = in.h(); p.in_bs = in.bs; p.in_Tp = in.Tp; p.in_coff8 = o.in_coff8;
  p.Tin = in.T; p.Cin = L.Cin; p.taps = L.taps; p.dil = L.dil; p.pad_left = L.pad_left;
  p.w = reinterpret_cast<const __half*>(blob + L.w_off); p.bias = blob + L.b_off; p.N = L.N; p.n_slices = L.n_slices; p.cta2 = L.cta2;
  p.mode = o.mode;
  p.out = out.h(); p.out_bs = out.bs; p.out_Tp = out.Tp; p.out_coff8 = o.out_coff8;
  p.Tout = o.Tout >= 0 ? o.Tout : out.T;
  if (o.pool) { p.pool = o.pool->h(); p.pool_bs = o.pool->bs; p.pool_Tp = o.pool->Tp; p.pool_coff8 = 0; }
  if (o.res) { p.res = o.res->h(); p.res_bs = o.res->bs; p.res_Tp = o.res->Tp; p.res_coff8 = 0; }
  p.lrelu = o.lrelu;
  p.out_tblock = o.out_tblock;
  p.B = B;
  p.tiles_per_item = (in.T + stride - 1) / stride;
  return p;
}

static int run_conv(Ctx& c, const std::string& name, const Act& in, const Act& out, const ConvOpt& o = ConvOpt()) {
  if (c.ar.dry) return AR_OK;
  auto it = c.m->conv.find(name);
  AR_CHECK(it != c.m->conv.end(), AR_ERR_INVALID, "internal: unknown conv layer " + name);
  const ConvLayer& L = it->second;
  const ConvParams p = conv_params(L, c.m->blob, in, out, o, c.B, TILE_M);
  {
    ProfScope ps(CAT_CONV, c.stream, 2.0 * L.macs_per_row * (double)c.B * (double)in.T);
    AR_TRY(c.m->engine == AR_ENGINE_SIMT ? launch_conv_simt(p, c.stream) : launch_conv_umma2(p, c.stream));
  }
  if (c.m->audit) {
    const int ncols = o.mode == MODE_INTERLEAVE2 ? L.N / 2 : L.N;
    AR_TRY(audit_act(c, name, out, o.out_coff8, ncols / 8, p.Tout, o.out_tblock));
    if (o.pool) AR_TRY(audit_act(c, name + ".pool", *o.pool, 0, ncols / 8, in.T / 2));
  }
  return AR_OK;
}

// A k-tap conv followed by one or two more convs as ONE fused launch (conv_chain.cu): pointwise follow-ups (the stereo
// `_dilated_block`, stereo_separator.py:49-64, and the LSTM input projection behind the last one) or one k3 follow-up (the
// U-Net double conv, denoiser.py:51-60, and the super-resolution residual block, super_resolution.py:104-122).  `o`
// describes the LAST stage's output (lrelu, layout, pool copy, residual operand); intermediate stages apply LeakyReLU.
static bool can_chain(const Ctx& c, std::initializer_list<const char*> names) {
  if (!c.m->fuse || c.m->audit || c.m->engine != AR_ENGINE_UMMA) return false;   // the audit looks at every intermediate
  bool first = true;
  int prevN = 0, Cin = 0, taps = 0, dil = 0, taps2 = 1, N[3] = {0, 0, 0}, ng = 0;
  for (const char* n : names) {
    auto it = c.m->conv.find(n);
    if (it == c.m->conv.end() || ng == 3) return false;
    const ConvLayer& L = it->second;
    if (!L.cta2 || L.n_slices != 2) return false;
    if (first) { Cin = L.Cin; taps = L.taps; dil = L.dil; }
    else {
      if (L.Cin != prevN || L.dil != 1) return false;
      if (ng == 1) taps2 = L.taps;
      else if (L.taps != 1) return false;
    }
    prevN = L.N;
    N[ng++] = L.N;
    first = false;
  }
  if (!conv_chain_fits(Cin, taps, dil, N, ng, taps2)) return false;
  // k3 -> k3 pairs (tile stride 126; tile groups of 2 / 4 for the narrow ones) are all faster fused than as two launches
  // (per 1184-chunk step, ncu: 32 -> 64 -> 64 + pool 1.77 vs 2.37 ms, 64 -> 128 -> 128 + pool 1.90 vs 2.40, 128 -> 64 -> 64 2.62 vs
  // 2.86, 64 -> 32 -> 32 2.14 vs 2.77; the super-resolution block 32 -> 32 -> 32 + skip ~1.9 vs 2.7 once its residual rows are
  // requested for a whole tile group ahead of the accumulator wait: model 17.5 vs 20.5 ms).  Without tile groups the narrow ones
  // lost (2.4 - 3.8 ms): profiles/README_r02.md.
  return true;
}

static int run_chain(Ctx& c, std::initializer_list<const char*> names, const Act& in, const Act& out, const ConvOpt& o = ConvOpt()) {
  if (c.ar.dry) return AR_OK;
  ChainParams cp;
  std::memset(&cp, 0, sizeof(cp));
  const ConvLayer* L[3];
  double macs = 0.0;
  int g = 0;
  for (const char* n : names) {
    L[g] = &c.m->conv.at(n);
    cp.w[g] = reinterpret_cast<const __half*>(c.m->blob + L[g]->w_off);
    cp.bias[g] = c.m->blob + L[g]->b_off;
    cp.N[g] = L[g]->N;
    cp.lrelu[g] = 1;
    macs += L[g]->macs_per_row;
    ++g;
  }
  cp.n_gemms = g;
  cp.taps2 = L[1]->taps;
  cp.lrelu[g - 1] = o.lrelu;
  const int stride = chain_tile_stride(cp.taps2);
  // the first stage is a plain conv with LeakyReLU (launch_conv_chain takes no other); `o` describes the last stage's output
  ConvOpt first;
  first.in_coff8 = o.in_coff8;
  cp.p = conv_params(*L[0], c.m->blob, in, out, first, c.B, stride);
  cp.pl = conv_params(*L[g - 1], c.m->blob, in, out, o, c.B, stride);
  cp.head_y = o.head_y;
  cp.head_xlr = o.head_xlr;
  long long* const trace = g_chain_trace.load();
  cp.trace = trace ? trace + (size_t)(g_chain_trace_slot.fetch_add(1) % 8) * 1024 : nullptr;
  ProfScope ps(CAT_CONV, c.stream, 2.0 * macs * (double)c.B * (double)in.T);
  return launch_conv_chain(cp, c.stream);
}

// Layers `names` in sequence from `cur` into `out`, `o` describing the last one's output and `o.in_coff8` the first one's
// input: one fused launch when the chain kernel takes them, else one launch per layer through intermediates as wide as each
// layer's N.  Without `out` the sequence consumes `cur` and leaves its output (as wide as the last layer) there: each tensor
// is then allocated when its layer runs and `cur` released once read, so layer by layer at most two are alive at a time.
static int run_seq(Ctx& c, std::initializer_list<const char*> names, Act& cur, const Act* out = nullptr, const ConvOpt& o = ConvOpt()) {
  const bool consume = out == nullptr;
  auto dst = [&](const char* n, bool last) { return last && !consume ? *out : c.ar.act(c.B, c.m->conv.at(n).N, cur.T); };
  if (can_chain(c, names)) {
    const Act y = dst(*(names.end() - 1), true);
    AR_TRY(run_chain(c, names, cur, y, o));
    if (consume) { c.ar.release(cur); cur = y; }
    return AR_OK;
  }
  Act x = cur;
  size_t k = 0;
  for (const char* n : names) {
    const bool first = k == 0, last = ++k == names.size();
    ConvOpt ok = last ? o : ConvOpt();
    ok.in_coff8 = first ? o.in_coff8 : 0;
    const Act y = dst(n, last);
    AR_TRY(run_conv(c, n, x, y, ok));
    if (!first || consume) c.ar.release(x);
    x = y;
  }
  if (consume) cur = x;
  return AR_OK;
}

// the stereo k7 output heads run on the tensor core (final_umma.cu) with the tcgen05 engine, on CUDA cores with the cross-check engine
static bool use_final_umma(const Model& m) { return m.engine == AR_ENGINE_UMMA; }

// ---------------------------------------------------------------------------- denoiser.py:88-144
static int denoiser_forward(Ctx& c, const float* x, float* y, int T) {
  AR_CHECK(T >= 8, AR_ERR_INVALID, "max_pool1d(): Invalid computed output size: 0 (denoiser needs at least 8 samples)");
  const Model& m = *c.m;
  const int B = c.B, T1 = T / 2, T2 = T1 / 2, T3 = T2 / 2;
  Arena& A = c.ar;
  Act e0a = A.act(B, 32, T), cat0 = A.act(B, 64, T), p0 = A.act(B, 32, T1);
  if (!A.dry) {
    ProfScope ps(CAT_STEM, c.stream, 2.0 * 96 * (double)B * T);
    AR_TRY(launch_stem(x, B, T, m.stem, e0a, 1, c.stream));
  }
  AR_TRY(audit_act(c, "stem", e0a, 0, 4, T));
  ConvOpt o; o.pool = &p0;
  AR_TRY(run_conv(c, "enc0b", e0a, cat0, o));                 // skip s0 -> cat0[0:32], pooled -> p0
  A.release(e0a);
  // levels 1, 2 and the three decoder levels: each double conv (denoiser.py:51-60) is ONE fused k3 -> k3 launch whose
  // intermediate stays in shared memory (the bottleneck's 256-channel intermediate does not fit: two launches)
  Act cat1 = A.act(B, 128, T1), p1 = A.act(B, 64, T2);
  o = ConvOpt(); o.pool = &p1;
  AR_TRY(run_seq(c, {"enc1a", "enc1b"}, p0, &cat1, o));
  A.release(p0);
  Act cat2 = A.act(B, 256, T2), p2 = A.act(B, 128, T3);
  o = ConvOpt(); o.pool = &p2;
  AR_TRY(run_seq(c, {"enc2a", "enc2b"}, p1, &cat2, o));
  A.release(p1);
  Act b1 = A.act(B, 256, T3);
  AR_TRY(run_seq(c, {"bot_a", "bot_b"}, p2, &b1));
  A.release(p2);
  // decoder level 0: up-conv writes the upper channel half of the concat buffer (skip first, :124)
  o = ConvOpt(); o.mode = MODE_INTERLEAVE2; o.lrelu = 0; o.out_coff8 = 128 / 8; o.Tout = T2;
  AR_TRY(run_conv(c, "up0", b1, cat2, o));
  A.release(b1);
  Act d0b = A.act(B, 128, T2);
  AR_TRY(run_seq(c, {"dec0a", "dec0b"}, cat2, &d0b));
  A.release(cat2);
  o = ConvOpt(); o.mode = MODE_INTERLEAVE2; o.lrelu = 0; o.out_coff8 = 64 / 8; o.Tout = T1;
  AR_TRY(run_conv(c, "up1", d0b, cat1, o));
  A.release(d0b);
  Act d1b = A.act(B, 64, T1);
  AR_TRY(run_seq(c, {"dec1a", "dec1b"}, cat1, &d1b));
  A.release(cat1);
  o = ConvOpt(); o.mode = MODE_INTERLEAVE2; o.lrelu = 0; o.out_coff8 = 32 / 8; o.Tout = T;
  AR_TRY(run_conv(c, "up2", d1b, cat0, o));
  A.release(d1b);
  Act f = A.act(B, 32, T);
  AR_TRY(run_seq(c, {"dec2a", "dec2b"}, cat0, &f));
  A.release(cat0);
  // the cross-check engine keeps the whole transient detector on CUDA cores
  if (c.m->engine == AR_ENGINE_UMMA) {
    Act h1 = A.act(B, 32, T);
    AR_TRY(run_conv(c, "td0", f, h1));
    if (!A.dry) {
      ProfScope ps(CAT_TAIL, c.stream, 2.0 * 440 * (double)B * T);
      AR_TRY(launch_den_tail(f, &h1, x, y, B, T, m.den_tail, c.stream));
    }
    A.release(h1);
  } else if (!A.dry) {
    ProfScope ps(CAT_TAIL, c.stream, 2.0 * 1976 * (double)B * T);
    AR_TRY(launch_den_tail(f, nullptr, x, y, B, T, m.den_tail, c.stream));
  }
  A.release(f);
  return AR_OK;
}

// ---------------------------------------------------------------------------- super_resolution.py:66-101
static int sr_forward(Ctx& c, const float* x, float* y, int T) {
  AR_CHECK(T >= 1, AR_ERR_INVALID, "super-resolution: empty input");
  const Model& m = *c.m;
  const int B = c.B;
  Arena& A = c.ar;
  Act f0 = A.act(B, 32, T);
  if (!A.dry) {
    ProfScope ps(CAT_STEM, c.stream, 2.0 * 224 * (double)B * T);
    AR_TRY(launch_stem(x, B, T, m.stem, f0, 1, c.stream));
  }
  AR_TRY(audit_act(c, "stem", f0, 0, 4, T));
  Act r = f0;
  static const char* const RA[4] = {"rb0a", "rb1a", "rb2a", "rb3a"};
  static const char* const RB[4] = {"rb0b", "rb1b", "rb2b", "rb3b"};
  for (int i = 0; i < 4; ++i) {
    // one residual block (conv-BN-LReLU-conv-BN + skip, super_resolution.py:104-122) = ONE fused k3 -> k3 launch; the
    // skip operand is the block's own input
    Act r2 = A.act(B, 32, T);
    ConvOpt o; o.lrelu = 0; o.res = &r;
    AR_TRY(run_seq(c, {RA[i], RB[i]}, r, &r2, o));
    if (i > 0) A.release(r);
    r = r2;
  }
  Act mid = A.act(B, 32, T);
  ConvOpt o; o.lrelu = 0; o.res = &f0;
  AR_TRY(run_conv(c, "middle", r, mid, o));
  A.release(r);
  A.release(f0);
  Act u = A.act(B, 32, 2 * T);
  o = ConvOpt(); o.mode = MODE_INTERLEAVE2; o.Tout = 2 * T;
  AR_TRY(run_conv(c, "up", mid, u, o));
  A.release(mid);
  if (can_chain(c, {"hf", "head"})) {
    // hf_emphasis (k5 + LeakyReLU) and the reconstruction head (k7 32 -> 1) + interpolation residual as ONE fused launch:
    // the 32-channel tensor at the output rate (128 B per output sample written + read back) never reaches HBM
    ConvOpt oh; oh.lrelu = 0; oh.head_y = y; oh.head_xlr = x; oh.Tout = 2 * T;
    AR_TRY(run_chain(c, {"hf", "head"}, u, u, oh));
    A.release(u);
    return AR_OK;
  }
  Act h = A.act(B, 32, 2 * T);
  AR_TRY(run_conv(c, "hf", u, h));
  A.release(u);
  if (!A.dry) {
    const int coff[1] = {0};
    ProfScope ps(CAT_TAIL, c.stream, 2.0 * 224 * (double)B * 2 * T);
    // one head = 8 KB of activations per tile: the tensor-core head kernel is latency-bound there (measured 3.0 ms per
    // 1184-chunk step against 2.5 ms of this CUDA-core kernel)
    AR_TRY(launch_final_k7(h, coff, m.fin, 1, y, B, 2 * T, x, c.stream));
  }
  A.release(h);
  return AR_OK;
}

// ---------------------------------------------------------------------------- stereo_separator.py:85-122
// The LSTM scan covers steps [w.lstm_start, T) (hidden states before it are zero) starting from `state_in`, and
// `state_out` receives (h, c) after step w.state_pos - 1: the window parameters of the whole-file-exact chunked mode
// (ar_stereo_forward_window), where a segment carries conv halos on both sides of the range whose state it hands on.
// With `cap` (device, [B]) item b hands its state on after step lstm_start + cap[b] - 1 instead, in the same launch
// (ar_stereo_forward_window_multi: windows of different files, each handing on at its own position).
struct LstmWindow { int lstm_start = 0, state_pos = -1; const int* cap = nullptr; };

// The forward in three phases, so that the chain (chain_forward below) can run them on different batch splits:
//   encode  stem + dilated encoder + LSTM input projection  x[B,1,T] -> xp (gate pre-activations, time-blocked fp16)
//   scan    the LSTM recurrence                             xp -> h
//   decode  both decoders + output heads                    h -> y[B,2,T]
// `xp` of stereo_encode: a tensor the caller allocated (base != nullptr), else it is allocated here, as late as possible.
// With `proj_in_scan` the scan kernel computes the input projection itself (lstm_proj.cu: batches beyond 8 sequences per SM)
// and `xp` is the encoder output e4b (128 channels, plain H8) instead of the 256 gate pre-activations.
static bool proj_in_scan(const Model& m, int B_scan) { return m.engine == AR_ENGINE_UMMA && m.fuse && !m.audit && B_scan > 8 * sm_count(); }

static int stereo_encode(Ctx& c, const float* x, int T, Act& xp, bool fused_proj) {
  const Model& m = *c.m;
  const int B = c.B;
  Arena& A = c.ar;
  const bool own_xp = xp.base == nullptr && xp.C == 0;
  Act cur = A.act(B, 32, T);
  if (!A.dry) {
    ProfScope ps(CAT_STEM, c.stream, 2.0 * 224 * (double)B * T);
    AR_TRY(launch_stem(x, B, T, m.stem, cur, 1, c.stream));
  }
  AR_TRY(audit_act(c, "stem", cur, 0, 4, T));
  // blocks 1-3 consume their input: beside a sub-batched chain's xp the encoder is the workspace peak
  AR_TRY(run_seq(c, {"enc1a", "enc1b"}, cur));
  AR_TRY(run_seq(c, {"enc2a", "enc2b"}, cur));
  AR_TRY(run_seq(c, {"enc3a", "enc3b"}, cur));
  ConvOpt oxp; oxp.lrelu = 0; oxp.out_tblock = 1;   // gate pre-activations, time-blocked: the recurrence streams 4 KB runs
  if (fused_proj) {
    if (own_xp) xp = A.act(B, 128, T);
    AR_TRY(run_seq(c, {"enc4a", "enc4b"}, cur, &xp));
  } else if (can_chain(c, {"enc4a", "enc4b", "xproj"})) {
    // last dilated block + LSTM input projection: 128 -k3 d8-> 128 -k1-> 128 -k1-> 256 in one launch
    if (own_xp) xp = A.act(B, 256, T);
    AR_TRY(run_chain(c, {"enc4a", "enc4b", "xproj"}, cur, xp, oxp));
  } else {
    // the projection is not part of the sequence: xp would be alive beside both 128-channel intermediates
    AR_TRY(run_seq(c, {"enc4a", "enc4b"}, cur));
    if (own_xp) xp = A.act(B, 256, T);   // fp16 storage costs < 0.1 dB, halves the LSTM's HBM stream
    AR_TRY(run_conv(c, "xproj", cur, xp, oxp));
  }
  A.release(cur);
  return AR_OK;
}

static int stereo_scan(Ctx& c, const Act& xp, const Act& h, int T, const float* state_in, float* state_out, const LstmWindow& w,
                       bool fused_proj) {
  if (c.ar.dry) return AR_OK;
  const Model& m = *c.m;
  const int B = c.B;
  ProfScope ps(CAT_LSTM, c.stream, 2.0 * (fused_proj ? 16384 + 32768 : 16384) * (double)B * (T - w.lstm_start), w.state_pos < T ? 2 : 1);
  // a scan over steps [t0, t1) is the same kernel on base pointers advanced by t0 rows (t0 % 8 == 0 keeps the 8-step
  // blocks of the time-blocked pre-activations aligned)
  auto scan = [&](int t0, int t1, const float* st_in, float* st_out, const int* cap = nullptr) {
    Act xs = xp, hs = h;
    hs.base = h.h() + (long long)t0 * 8;
    xs.T = hs.T = t1 - t0;
    if (fused_proj) {
      xs.base = xp.h() + (long long)t0 * 8;
      return launch_lstm_proj(xs, reinterpret_cast<const __half*>(m.blob + m.wih_umma_off), m.blob + m.conv.at("xproj").b_off,
                              m.blob + m.whh_off, hs, B, t1 - t0, st_in, st_out, cap, c.stream);
    }
    xs.base = xp.h() + (long long)(t0 / 8) * 32 * 64;
    return launch_lstm(xs, m.blob + m.whh_off, hs, B, t1 - t0, st_in, st_out, cap, c.stream);
  };
  if (w.lstm_start > 0)   // rows [0, lstm_start) of all 8 chunks of every item: zero hidden states
    AR_CUDA_OK(cudaMemset2DAsync(h.h() + (long long)HALO * 8, (size_t)h.Tp * 16, 0, (size_t)w.lstm_start * 16, (size_t)B * 8, c.stream));
  if (w.cap != nullptr) {
    AR_CHECK(state_out != nullptr, AR_ERR_INVALID, "stereo: per-item state positions need state_out");
    AR_TRY(scan(w.lstm_start, T, state_in, state_out, w.cap));
  } else if (w.state_pos < T) {
    AR_CHECK(state_out != nullptr, AR_ERR_INVALID, "stereo: an interior state_pos needs state_out");
    AR_TRY(scan(w.lstm_start, w.state_pos, state_in, state_out));
    AR_TRY(scan(w.state_pos, T, state_out, nullptr));
  } else {
    AR_TRY(scan(w.lstm_start, T, state_in, state_out));
  }
  return AR_OK;
}

// `h_owned`: h is an arena tensor of this batch and is released as soon as the first layer has consumed it
static int stereo_decode(Ctx& c, const Act& h, float* y, int T, bool h_owned) {
  const Model& m = *c.m;
  const int B = c.B;
  Arena& A = c.ar;
  Act d0 = A.act(B, 256, T);
  AR_TRY(run_conv(c, "dec0", h, d0));
  if (h_owned) A.release(h);
  // per side: decoder layers 3 and 6 (128 -> 64 -> 32, both k7) as ONE fused k7 -> k7 launch when the chain kernel has them
  // (the 64-channel intermediate stays in shared memory), else two launches through a 64-channel tensor
  Act d2 = A.act(B, 64, T);
  ConvOpt o;
  AR_TRY(run_seq(c, {"dec1L", "dec2L"}, d0, &d2, o));
  o.in_coff8 = 128 / 8; o.out_coff8 = 32 / 8;
  AR_TRY(run_seq(c, {"dec1R", "dec2R"}, d0, &d2, o));
  A.release(d0);
  if (!A.dry) {
    const int coff[2] = {0, 32 / 8};
    ProfScope ps(CAT_TAIL, c.stream, 2.0 * 448 * (double)B * T);
    if (use_final_umma(m))
      AR_TRY(launch_final_umma(d2, 0, reinterpret_cast<const __half*>(m.blob + m.fin_umma_off), m.fin, 2, y, B, T, nullptr, c.stream));
    else
      AR_TRY(launch_final_k7(d2, coff, m.fin, 2, y, B, T, nullptr, c.stream));
  }
  A.release(d2);
  return AR_OK;
}

static int check_window(LstmWindow& w, int T) {
  AR_CHECK(T >= 1, AR_ERR_INVALID, "stereo: empty input");
  if (w.state_pos < 0) w.state_pos = T;
  AR_CHECK(w.lstm_start >= 0 && w.lstm_start < w.state_pos && w.state_pos <= T && w.lstm_start % 8 == 0 &&
               (w.state_pos % 8 == 0 || w.state_pos == T),
           AR_ERR_INVALID, "stereo: LSTM window must satisfy 0 <= lstm_start < state_pos <= T, both multiples of 8 (state_pos may be T)");
  return AR_OK;
}

static int stereo_forward(Ctx& c, const float* x, float* y, int T, const float* state_in, float* state_out,
                          LstmWindow w = LstmWindow()) {
  AR_TRY(check_window(w, T));
  Arena& A = c.ar;
  const bool fp = proj_in_scan(*c.m, c.B);
  Act xp{};
  AR_TRY(stereo_encode(c, x, T, xp, fp));
  Act h = A.act(c.B, 64, T);
  AR_TRY(stereo_scan(c, xp, h, T, state_in, state_out, w, fp));
  AR_TRY(audit_act(c, "lstm", h, 0, 64 / 8, T));
  A.release(xp);
  return stereo_decode(c, h, y, T, true);
}

// ---------------------------------------------------------------------------- inference.py:59-95, chunk batches
// denoise -> super-resolve -> stereo on B independent chunks.  Up to 8 chunks per SM the three forwards run one after the
// other on the whole batch.  Beyond that the batch exists for the LSTM's sake -- its recurrence is a latency chain per
// sequence, and 16 sequences per SM (lstm_mmaw_kernel<8>) cost barely more per step than 8 -- while the convs gain nothing
// from it and their activations (45 - 68 MB per chunk) would not fit: so the conv phases run on sub-batches around ONE scan,
//   for each sub-batch:  denoiser, super-resolution, stereo encoder  ->  its slice of the gate pre-activations xp
//   LSTM scan over all B sequences                                    ->  h
//   for each sub-batch:  decoders                                     ->  its slice of y
// and the workspace holds the scan's input (the encoder output, 23 MB per chunk: the scan kernel of such batches computes
// the LSTM input projection itself, lstm_proj.cu) / h (11 MB per chunk) for the batch plus the conv scratch of one sub-batch.
static int chain_run(Ctx& c, const Model* den, const Model* sr, const Model* st, const float* x, float* y, int B, int T) {
  Arena& A = c.ar;
  const int rate = sr ? 2 : 1, Ts = rate * T;
  const int full = 8 * sm_count();
  const bool fp = proj_in_scan(*st, B);
  // sub-batches: 8 per SM; 4 per SM in front of a scan that reads stored pre-activations (256 channels for the whole batch
  // leave less room for the encoder's scratch)
  const int sub_front = B <= full ? B : (fp ? full : full / 2), sub_back = B <= full ? B : full;
  auto front = [&](int b0, int nb, Act& xp) {      // chunks [b0, b0 + nb) -> xp (allocated inside when xp is empty)
    c.B = nb;
    float* y1 = A.plain((size_t)nb * T);
    c.m = den;
    AR_TRY(denoiser_forward(c, x + (size_t)b0 * T, y1, T));
    const float* st_in = y1;
    float* y2 = nullptr;
    if (sr) {
      y2 = A.plain((size_t)nb * Ts);
      c.m = sr;
      AR_TRY(sr_forward(c, y1, y2, T));
      A.release_plain(y1);
      st_in = y2;
    }
    c.m = st;
    AR_TRY(stereo_encode(c, st_in, Ts, xp, fp));
    A.release_plain(sr ? y2 : y1);
    return (int)AR_OK;
  };
  LstmWindow w;
  AR_TRY(check_window(w, Ts));
  if (B <= full) {
    Act xp{};
    AR_TRY(front(0, B, xp));
    Act h = A.act(B, 64, Ts);
    AR_TRY(stereo_scan(c, xp, h, Ts, nullptr, nullptr, w, fp));
    A.release(xp);
    return stereo_decode(c, h, y, Ts, true);
  }
  Act xp = A.act(B, fp ? 128 : 256, Ts);
  for (int b0 = 0; b0 < B; b0 += sub_front) {
    Act v = xp;
    v.base = xp.h() + (long long)b0 * xp.bs;
    AR_TRY(front(b0, std::min(sub_front, B - b0), v));
  }
  Act h = A.act(B, 64, Ts);
  c.m = st;
  c.B = B;
  AR_TRY(stereo_scan(c, xp, h, Ts, nullptr, nullptr, w, fp));
  A.release(xp);
  for (int b0 = 0; b0 < B; b0 += sub_back) {
    Act v = h;
    v.base = h.h() + (long long)b0 * h.bs;
    c.B = std::min(sub_back, B - b0);
    AR_TRY(stereo_decode(c, v, y + (size_t)b0 * 2 * Ts, Ts, false));
  }
  A.release(h);
  return AR_OK;
}

int chain_workspace_bytes(const Model* den, const Model* sr, const Model* st, int B, int T, size_t* bytes) {
  AR_CHECK(den && st && bytes && B >= 1 && T >= 1, AR_ERR_INVALID, "chain: bad argument");
  Ctx c;
  c.ar.dry = true;
  AR_TRY(chain_run(c, den, sr, st, nullptr, nullptr, B, T));
  *bytes = c.ar.peak + 256;
  return AR_OK;
}

int chain_forward(const Model* den, const Model* sr, const Model* st, const float* x, float* y, int B, int T, void* ws,
                  size_t ws_bytes, cudaStream_t stream) {
  AR_CHECK(x && y, AR_ERR_INVALID, "chain: null tensor");
  size_t need = 0;
  AR_TRY(chain_workspace_bytes(den, sr, st, B, T, &need));
  AR_CHECK(ws != nullptr && ws_bytes >= need, AR_ERR_WORKSPACE, "chain: workspace too small (need " + std::to_string(need) + " bytes)");
  Ctx c;
  c.stream = stream;
  c.ar.dry = false;
  c.ar.base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) / 256 * 256);
  c.ar.cap = need - 256;        // == the dry-run peak: high-side tensors are placed down from it
  return chain_run(c, den, sr, st, x, y, B, T);
}

static int dispatch(Ctx& c, const float* x, float* y, int T, const float* st_in, float* st_out, LstmWindow w = LstmWindow()) {
  switch (c.m->kind) {
    case AR_MODEL_DENOISER: return denoiser_forward(c, x, y, T);
    case AR_MODEL_SUPER_RES: return sr_forward(c, x, y, T);
    case AR_MODEL_STEREO: return stereo_forward(c, x, y, T, st_in, st_out, w);
  }
  set_error("internal: bad model kind");
  return AR_ERR_INVALID;
}

// A stereo forward's workspace ends with room for B per-item LSTM state positions (ar_stereo_forward_window_multi)
static size_t cap_bytes(const Model* m, int B) { return m->kind == AR_MODEL_STEREO ? ((size_t)B * sizeof(int) + 255) / 256 * 256 : 0; }

int model_workspace_bytes(const Model* m, int B, int T, size_t* bytes) {
  AR_CHECK(m && bytes && B >= 1 && T >= 1, AR_ERR_INVALID, "workspace_bytes: bad argument");
  Ctx c;
  c.m = m; c.B = B; c.ar.dry = true;
  AR_TRY(dispatch(c, nullptr, nullptr, T, nullptr, nullptr));
  *bytes = c.ar.peak + 256 + cap_bytes(m, B);
  return AR_OK;
}

int model_forward(const Model* m, const float* x, float* y, int B, int T, const float* st_in, float* st_out, void* ws,
                  size_t ws_bytes, cudaStream_t stream, int lstm_start, int state_pos, const int* state_pos_host) {
  AR_CHECK(m && x && y && B >= 1 && T >= 1, AR_ERR_INVALID, "forward: bad argument");
  size_t need = 0;
  AR_TRY(model_workspace_bytes(m, B, T, &need));
  AR_CHECK(ws != nullptr && ws_bytes >= need, AR_ERR_WORKSPACE, "forward: workspace too small (need " + std::to_string(need) + " bytes)");
  Ctx c;
  c.m = m; c.B = B; c.stream = stream;
  c.ar.dry = false;
  uintptr_t a = (reinterpret_cast<uintptr_t>(ws) + 255) / 256 * 256;
  c.ar.base = reinterpret_cast<char*>(a);
  c.ar.cap = need - 256 - cap_bytes(m, B);   // == the dry-run peak: high-side tensors are placed down from it
  LstmWindow w;
  w.lstm_start = lstm_start;
  w.state_pos = state_pos;
  if (state_pos_host != nullptr) {
    AR_CHECK(m->kind == AR_MODEL_STEREO && st_out != nullptr, AR_ERR_INVALID, "forward: per-item state positions need a stereo model and state_out");
    std::vector<int> local(B);
    for (int b = 0; b < B; ++b) {
      AR_CHECK(lstm_start < state_pos_host[b] && state_pos_host[b] <= T, AR_ERR_INVALID,
               "stereo: state_pos[" + std::to_string(b) + "] = " + std::to_string(state_pos_host[b]) +
                   " must satisfy lstm_start < state_pos <= T");
      local[b] = state_pos_host[b] - lstm_start;   // the scan kernels count steps from lstm_start
    }
    int* dcap = reinterpret_cast<int*>(c.ar.base + c.ar.cap);
    // pageable source: staged before the call returns, so `local` may go; no host sync
    AR_CUDA_OK(cudaMemcpyAsync(dcap, local.data(), (size_t)B * sizeof(int), cudaMemcpyHostToDevice, stream));
    w.cap = dcap;
    w.state_pos = T;
  }
  return dispatch(c, x, y, T, st_in, st_out, w);
}

// ---------------------------------------------------------------------------- dynamic-range audit (ar_model_audit_*)
int model_audit_enable(Model* m, int on) {
  AR_CHECK(m != nullptr, AR_ERR_INVALID, "audit: null model");
  if (on && m->audit_dev == nullptr) {
    AR_CUDA_OK(cudaSetDevice(m->device));
    AR_CUDA_OK(cudaMalloc(&m->audit_dev, AUDIT_SLOTS * sizeof(unsigned int)));
  }
  if (on) {
    AR_CUDA_OK(cudaSetDevice(m->device));
    AR_CUDA_OK(cudaMemset(m->audit_dev, 0, AUDIT_SLOTS * sizeof(unsigned int)));
    AR_CUDA_OK(cudaDeviceSynchronize());   // diagnostic path: the clear is complete before launches on any stream
    m->audit_names.clear();
  }
  m->audit = on != 0;
  return AR_OK;
}
// Synchronises the device; max_abs[i] / name(i) describe the i-th audited tensor since the audit was enabled.
int model_audit_read(Model* m, float* max_abs, int cap, int* n_layers) {
  AR_CHECK(m && max_abs && n_layers && cap >= 1, AR_ERR_INVALID, "audit: bad argument");
  AR_CHECK(m->audit_dev != nullptr, AR_ERR_INVALID, "audit: not enabled for this model");
  AR_CUDA_OK(cudaSetDevice(m->device));
  AR_CUDA_OK(cudaDeviceSynchronize());
  unsigned int bits[AUDIT_SLOTS];
  AR_CUDA_OK(cudaMemcpy(bits, m->audit_dev, sizeof(bits), cudaMemcpyDeviceToHost));
  const int n = (int)m->audit_names.size();
  *n_layers = n;
  for (int i = 0; i < n && i < cap; ++i) std::memcpy(&max_abs[i], &bits[i], 4);
  return AR_OK;
}
const char* model_audit_name(const Model* m, int i) {
  return (m && i >= 0 && i < (int)m->audit_names.size()) ? m->audit_names[i].c_str() : nullptr;
}
int model_audit_tap(Model* m, const char* name, float* y, long long cap_floats) {
  AR_CHECK(m != nullptr, AR_ERR_INVALID, "audit tap: null model");
  if (name == nullptr) { m->audit_taps.clear(); return AR_OK; }
  AR_CHECK(y != nullptr && cap_floats >= 0, AR_ERR_INVALID, "audit tap: null buffer or negative capacity");
  m->audit_taps[name] = Model::Tap{y, cap_floats};
  return AR_OK;
}

void model_destroy(Model* m) { delete m; }
int model_kind(const Model* m) { return m->kind; }

// One conv layer through a chosen engine on plain [B,C,T] tensors (test hook, ar_debug_conv1d).
int debug_conv(const float* x, const float* w_host, const float* bias_host, float* y, int B, int Cin, int Cout, int T, int k,
               int dil, int lrelu, int engine, cudaStream_t stream) {
  AR_CHECK(x && w_host && bias_host && y && B >= 1 && T >= 1, AR_ERR_INVALID, "debug_conv: bad argument");
  AR_CHECK(Cin % 16 == 0 && Cout % 16 == 0 && Cout <= 256 && (k & 1) == 1 && dil * (k - 1) / 2 <= HALO, AR_ERR_INVALID,
           "debug_conv: unsupported shape");
  AR_CHECK(engine == AR_ENGINE_SIMT || Cout % 32 == 0, AR_ERR_INVALID, "debug_conv: the tcgen05 engine needs Cout % 32 == 0");
  Gemm g;
  g.init(Cin, Cout, k, dil, dil * (k - 1) / 2);
  for (int o = 0; o < Cout; ++o) {
    for (int c = 0; c < Cin; ++c)
      for (int j = 0; j < k; ++j) g.at(j, c, o) = w_host[((size_t)o * Cin + c) * k + j];
    g.bias[o] = bias_host[o];
  }
  Blob blob;
  ConvLayer L = blob.push_gemm(g);
  Arena D;
  D.dry = true;
  D.act(B, Cin, T);
  D.act(B, Cout, T);
  float* dblob = nullptr;
  char* dws = nullptr;
  AR_CUDA_OK(cudaMalloc(&dblob, blob.host.size() * sizeof(float)));
  AR_CUDA_OK(cudaMalloc(&dws, D.peak));
  AR_CUDA_OK(cudaMemcpyAsync(dblob, blob.host.data(), blob.host.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
  Arena A;
  A.dry = false;
  A.base = dws;
  A.cap = D.peak;
  Act in = A.act(B, Cin, T), out = A.act(B, Cout, T);
  int rc = launch_plain_to_c4(x, B, Cin, T, in, stream);
  if (rc == AR_OK) {
    ConvOpt o;
    o.lrelu = lrelu;
    const ConvParams p = conv_params(L, dblob, in, out, o, B, TILE_M);
    rc = engine == AR_ENGINE_SIMT ? launch_conv_simt(p, stream) : launch_conv_umma2(p, stream);
  }
  if (rc == AR_OK) rc = launch_c4_to_plain(out, B, Cout, T, y, stream);
  cudaError_t e = cudaStreamSynchronize(stream);
  cudaFree(dblob);
  cudaFree(dws);
  if (rc == AR_OK && e != cudaSuccess) { set_error(std::string("debug_conv: ") + cudaGetErrorString(e)); rc = AR_ERR_CUDA; }
  return rc;
}

}  // namespace ar
