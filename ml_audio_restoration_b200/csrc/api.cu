// extern "C" surface of libaudiorestore_sm100.so (see include/audiorestore.h).
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "ar_common.cuh"
#include "pointwise.cuh"
#include "prof.cuh"

namespace ar {
struct Model;
const char* last_error();
int set_engine(int e);
int set_fusion(int on);
int set_chain_trace(long long* dev_buf);
long long resample_length(long long n, int orig_sr, int new_sr);
int launch_resample_mono(const float* x, int channels, long long n, int orig_sr, int new_sr, float* y, long long n_out,
                         cudaStream_t stream);
int launch_pcm16(const short* pcm, int channels, long long n, float* y, cudaStream_t stream);
int launch_pcm_decode(const void* raw, int format, int channels, long long n, float* y, cudaStream_t stream);
int flac_workspace_bytes(long long nbytes, size_t* bytes);
int flac_decode(const unsigned char* data, long long nbytes, int channels, int bps, int sample_rate, int min_block,
                int max_block, long long total_samples, float* y, long long n, long long* n_out, void* ws, size_t ws_bytes,
                cudaStream_t stream);
int flac_encode_workspace_bytes(int channels, long long n, int block_size, int bps, size_t* workspace, size_t* out_capacity);
int flac_encode(const float* x, int channels, long long n, int bps, int sample_rate, int block_size, unsigned char* frames_out,
                size_t out_capacity, unsigned char* pcm_le_out, long long* frame_bytes_total, int* min_frame, int* max_frame,
                void* ws, size_t ws_bytes, cudaStream_t stream);
int butter(int order, double wn, int highpass, double* b, double* a);
int launch_vinyl_mix(const float* audio, const float* noise, float level, const void* pops, int n_pops, int sample_rate,
                     float* y, int rows, long long n, cudaStream_t stream);
int launch_vinyl_sum(const float* x0, const float* x1, const float* x2, float* y, long long count, cudaStream_t stream);
int filtfilt_workspace_bytes(int rows, long long n, int order, size_t* bytes);
int launch_filtfilt(const float* x, float scale, const float* add1, const float* add2, float* y, int rows, long long n,
                    const double* b, const double* a, int order, void* ws, size_t ws_bytes, cudaStream_t stream);
int model_create(int kind, const ar_tensor_t* tensors, int n, int device, Model** out);
int model_workspace_bytes(const Model* m, int B, int T, size_t* bytes);
int model_forward(const Model* m, const float* x, float* y, int B, int T, const float* st_in, float* st_out, void* ws,
                  size_t ws_bytes, cudaStream_t stream, int lstm_start = 0, int state_pos = -1,
                  const int* state_pos_host = nullptr);
int chain_workspace_bytes(const Model* den, const Model* sr, const Model* st, int B, int T, size_t* bytes);
int chain_forward(const Model* den, const Model* sr, const Model* st, const float* x, float* y, int B, int T, void* ws,
                  size_t ws_bytes, cudaStream_t stream);
void model_destroy(Model* m);
int model_kind(const Model* m);
int model_audit_enable(Model* m, int on);
int model_audit_read(Model* m, float* max_abs, int cap, int* n_layers);
const char* model_audit_name(const Model* m, int i);
int model_audit_tap(Model* m, const char* name, float* y, long long cap_floats);
int debug_conv(const float* x, const float* w_host, const float* bias_host, float* y, int B, int Cin, int Cout, int T, int k,
               int dil, int lrelu, int engine, cudaStream_t stream);
}  // namespace ar

struct ar_model_s;  // == ar::Model
struct ar_chain_s {
  ar::Model* den;
  ar::Model* sr;
  ar::Model* st;
};


extern "C" {

const char* ar_last_error(void) { return ar::last_error(); }
int ar_version(void) { return 100; }
int ar_set_conv_engine(int engine) { return ar::set_engine(engine); }
int ar_set_fusion(int on) { return ar::set_fusion(on); }
int ar_resample_length(int64_t n, int orig_sr, int new_sr, int64_t* n_out) {
  if (!n_out || n < 0 || orig_sr < 1 || new_sr < 1) { ar::set_error("resample_length: bad argument"); return AR_ERR_INVALID; }
  *n_out = ar::resample_length(n, orig_sr, new_sr);
  return AR_OK;
}
int ar_resample_mono(const float* x, int channels, int64_t n, int orig_sr, int new_sr, float* y, int64_t n_out, void* stream) {
  return ar::launch_resample_mono(x, channels, n, orig_sr, new_sr, y, n_out, reinterpret_cast<cudaStream_t>(stream));
}
int ar_pcm16_to_float(const int16_t* pcm, int channels, int64_t n, float* y, void* stream) {
  return ar::launch_pcm16(pcm, channels, n, y, reinterpret_cast<cudaStream_t>(stream));
}
int ar_pcm_to_float(const void* raw, int format, int channels, int64_t n, float* y, void* stream) {
  return ar::launch_pcm_decode(raw, format, channels, n, y, reinterpret_cast<cudaStream_t>(stream));
}
int ar_flac_workspace_bytes(int64_t nbytes, size_t* bytes) { return ar::flac_workspace_bytes(nbytes, bytes); }
int ar_flac_decode(const uint8_t* frames, int64_t nbytes, int channels, int bps, int sample_rate, int min_block, int max_block,
                   int64_t total_samples, float* y, int64_t n, int64_t* n_out, void* workspace, size_t workspace_bytes,
                   void* stream) {
  long long got = 0;
  const int rc = ar::flac_decode(frames, nbytes, channels, bps, sample_rate, min_block, max_block, total_samples, y, n, &got,
                                 workspace, workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
  if (n_out) *n_out = got;
  return rc;
}
int ar_flac_encode_workspace_bytes(int channels, int64_t n, int block_size, int bps, size_t* workspace, size_t* out_capacity) {
  return ar::flac_encode_workspace_bytes(channels, n, block_size, bps, workspace, out_capacity);
}
int ar_flac_encode(const float* x, int channels, int64_t n, int bps, int sample_rate, int block_size, uint8_t* frames_out,
                   size_t out_capacity, uint8_t* pcm_le_out, int64_t* frame_bytes_total, int* min_frame, int* max_frame,
                   void* workspace, size_t workspace_bytes, void* stream) {
  long long total = 0;
  const int rc = ar::flac_encode(x, channels, n, bps, sample_rate, block_size, frames_out, out_capacity, pcm_le_out, &total,
                                 min_frame, max_frame, workspace, workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
  if (frame_bytes_total) *frame_bytes_total = total;
  return rc;
}
int ar_butter(int order, double wn, int highpass, double* b, double* a) { return ar::butter(order, wn, highpass, b, a); }
int ar_vinyl_mix(const float* audio, const float* surface_noise, float surface_level, const ar_pop_t* pops, int n_pops,
                 int sample_rate, float* y, int rows, int64_t n, void* stream) {
  static_assert(sizeof(ar_pop_t) == 48, "ar_pop_t layout");
  return ar::launch_vinyl_mix(audio, surface_noise, surface_level, pops, n_pops, sample_rate, y, rows, n,
                              reinterpret_cast<cudaStream_t>(stream));
}
int ar_vinyl_sum(const float* x0, const float* x1, const float* x2, float* y, int64_t count, void* stream) {
  return ar::launch_vinyl_sum(x0, x1, x2, y, count, reinterpret_cast<cudaStream_t>(stream));
}
int ar_filtfilt_workspace_bytes(int rows, int64_t n, int order, size_t* bytes) {
  return ar::filtfilt_workspace_bytes(rows, n, order, bytes);
}
int ar_filtfilt(const float* x, float scale, const float* add1, const float* add2, float* y, int rows, int64_t n,
                const double* b, const double* a, int order, void* workspace, size_t workspace_bytes, void* stream) {
  return ar::launch_filtfilt(x, scale, add1, add2, y, rows, n, b, a, order, workspace, workspace_bytes,
                             reinterpret_cast<cudaStream_t>(stream));
}
int ar_debug_chain_trace(long long* dev_buf) { return ar::set_chain_trace(dev_buf); }

int ar_model_create(int kind, const ar_tensor_t* tensors, int n_tensors, int device, ar_model_t* out) {
  ar::Model* m = nullptr;
  int r = ar::model_create(kind, tensors, n_tensors, device, &m);
  if (r == AR_OK) *out = reinterpret_cast<ar_model_t>(m);
  return r;
}
void ar_model_destroy(ar_model_t m) { ar::model_destroy(reinterpret_cast<ar::Model*>(m)); }
int ar_model_kind(ar_model_t m) { return m ? ar::model_kind(reinterpret_cast<ar::Model*>(m)) : -1; }

int ar_model_audit_enable(ar_model_t m, int on) { return ar::model_audit_enable(reinterpret_cast<ar::Model*>(m), on); }
int ar_model_audit_read(ar_model_t m, float* max_abs, int cap, int* n_layers) {
  return ar::model_audit_read(reinterpret_cast<ar::Model*>(m), max_abs, cap, n_layers);
}
const char* ar_model_audit_name(ar_model_t m, int i) { return ar::model_audit_name(reinterpret_cast<ar::Model*>(m), i); }
int ar_model_audit_tap(ar_model_t m, const char* name, float* y, int64_t cap_floats) {
  return ar::model_audit_tap(reinterpret_cast<ar::Model*>(m), name, y, cap_floats);
}

int ar_model_workspace_bytes(ar_model_t m, int B, int T, size_t* bytes) {
  return ar::model_workspace_bytes(reinterpret_cast<ar::Model*>(m), B, T, bytes);
}

int ar_model_forward(ar_model_t m, const float* x, float* y, int B, int T, void* workspace, size_t workspace_bytes, void* stream) {
  return ar::model_forward(reinterpret_cast<ar::Model*>(m), x, y, B, T, nullptr, nullptr, workspace, workspace_bytes,
                           reinterpret_cast<cudaStream_t>(stream));
}

int ar_stereo_forward_state(ar_model_t m, const float* x, float* y, int B, int T, const float* state_in, float* state_out,
                            void* workspace, size_t workspace_bytes, void* stream) {
  AR_CHECK(m && ar::model_kind(reinterpret_cast<ar::Model*>(m)) == AR_MODEL_STEREO, AR_ERR_INVALID,
           "ar_stereo_forward_state: not a stereo model");
  return ar::model_forward(reinterpret_cast<ar::Model*>(m), x, y, B, T, state_in, state_out, workspace, workspace_bytes,
                           reinterpret_cast<cudaStream_t>(stream));
}

int ar_stereo_forward_window(ar_model_t m, const float* x, float* y, int B, int T, int lstm_start, int state_pos,
                             const float* state_in, float* state_out, void* workspace, size_t workspace_bytes, void* stream) {
  AR_CHECK(m && ar::model_kind(reinterpret_cast<ar::Model*>(m)) == AR_MODEL_STEREO, AR_ERR_INVALID,
           "ar_stereo_forward_window: not a stereo model");
  return ar::model_forward(reinterpret_cast<ar::Model*>(m), x, y, B, T, state_in, state_out, workspace, workspace_bytes,
                           reinterpret_cast<cudaStream_t>(stream), lstm_start, state_pos);
}

int ar_stereo_forward_window_multi(ar_model_t m, const float* x, float* y, int B, int T, int lstm_start, const int* state_pos,
                                   const float* state_in, float* state_out, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  AR_CHECK(m && ar::model_kind(reinterpret_cast<ar::Model*>(m)) == AR_MODEL_STEREO, AR_ERR_INVALID,
           "ar_stereo_forward_window_multi: not a stereo model");
  AR_CHECK(state_pos != nullptr, AR_ERR_INVALID, "ar_stereo_forward_window_multi: null state_pos");
  return ar::model_forward(reinterpret_cast<ar::Model*>(m), x, y, B, T, state_in, state_out, workspace, workspace_bytes,
                           reinterpret_cast<cudaStream_t>(stream), lstm_start, -1, state_pos);
}

int ar_chain_create(ar_model_t denoiser, ar_model_t sr, ar_model_t stereo, ar_chain_t* out) {
  AR_CHECK(out && denoiser && stereo, AR_ERR_INVALID, "ar_chain_create: denoiser and stereo models are required");
  AR_CHECK(ar_model_kind(denoiser) == AR_MODEL_DENOISER && ar_model_kind(stereo) == AR_MODEL_STEREO &&
               (sr == nullptr || ar_model_kind(sr) == AR_MODEL_SUPER_RES),
           AR_ERR_INVALID, "ar_chain_create: model kinds do not match their slots");
  ar_chain_s* c = new ar_chain_s;
  c->den = reinterpret_cast<ar::Model*>(denoiser);
  c->sr = reinterpret_cast<ar::Model*>(sr);
  c->st = reinterpret_cast<ar::Model*>(stereo);
  *out = c;
  return AR_OK;
}
void ar_chain_destroy(ar_chain_t c) { delete c; }

int ar_chain_workspace_bytes(ar_chain_t c, int B, int T, size_t* bytes) {
  AR_CHECK(c != nullptr, AR_ERR_INVALID, "chain: null handle");
  return ar::chain_workspace_bytes(c->den, c->sr, c->st, B, T, bytes);
}

int ar_chain_forward(ar_chain_t c, const float* x, float* y, int B, int T, void* workspace, size_t workspace_bytes, void* stream) {
  AR_CHECK(c != nullptr, AR_ERR_INVALID, "chain: null handle");
  return ar::chain_forward(c->den, c->sr, c->st, x, y, B, T, workspace, workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
}

int ar_normalize(float* audio, int64_t n, float target_db, void* scratch, void* stream) {
  AR_CHECK(audio && scratch, AR_ERR_INVALID, "ar_normalize: null pointer");
  ar::ProfScope ps(ar::CAT_NORM, reinterpret_cast<cudaStream_t>(stream), 0.0, 2);
  return ar::launch_normalize(audio, n, target_db, reinterpret_cast<float*>(scratch), reinterpret_cast<cudaStream_t>(stream));
}

int ar_num_chunks(int64_t n, int chunk_size, int overlap, int* n_chunks) {
  AR_CHECK(n_chunks != nullptr, AR_ERR_INVALID, "ar_num_chunks: null output");
  AR_CHECK(chunk_size > 0 && overlap >= 0 && overlap <= chunk_size / 2, AR_ERR_INVALID, "overlap must be in [0, chunk_size // 2]");
  AR_CHECK(n > 0, AR_ERR_INVALID, "empty audio");
  const int64_t hop = chunk_size - overlap;
  const int64_t k = n <= chunk_size ? 1 : (n - overlap + hop - 1) / hop;
  AR_CHECK(k < (1LL << 31), AR_ERR_INVALID, "too many chunks");
  *n_chunks = (int)k;
  return AR_OK;
}

int ar_split_chunks(const float* audio, int64_t n, float* chunks, int first, int count, int chunk_size, int overlap, void* stream) {
  int total = 0;
  AR_TRY(ar_num_chunks(n, chunk_size, overlap, &total));
  AR_CHECK(audio && chunks && first >= 0 && count >= 0 && first + count <= total, AR_ERR_INVALID, "ar_split_chunks: bad chunk range");
  ar::ProfScope ps(ar::CAT_CHUNK, reinterpret_cast<cudaStream_t>(stream), 0.0);
  return ar::launch_split(audio, n, chunks, first, count, chunk_size, overlap, reinterpret_cast<cudaStream_t>(stream));
}

int ar_overlap_add(const float* y, float* out, int64_t n, int n_chunks, int channels, int chunk_size, int overlap, int rate,
                   void* stream) {
  int total = 0;
  AR_TRY(ar_num_chunks(n, chunk_size, overlap, &total));
  AR_CHECK(y && out && n_chunks == total && channels >= 1 && rate >= 1, AR_ERR_INVALID, "ar_overlap_add: bad argument");
  ar::ProfScope ps(ar::CAT_CHUNK, reinterpret_cast<cudaStream_t>(stream), 0.0);
  return ar::launch_ola(y, out, n, n_chunks, channels, chunk_size, overlap, rate, reinterpret_cast<cudaStream_t>(stream));
}

int ar_gather_windows(const float* src, int64_t src_len, const int64_t* offsets, int B, int W, float* dst, void* workspace,
                      size_t workspace_bytes, void* stream) {
  ar::ProfScope ps(ar::CAT_CHUNK, reinterpret_cast<cudaStream_t>(stream), 0.0);
  return ar::launch_gather_windows(src, src_len, reinterpret_cast<const long long*>(offsets), B, W, dst, workspace, workspace_bytes,
                                   reinterpret_cast<cudaStream_t>(stream));
}

int ar_scatter_kept(const float* y, int B, int W, const int64_t* dst_offsets, const int* lo, const int* len, float* out,
                    int64_t out_len, void* workspace, size_t workspace_bytes, void* stream) {
  ar::ProfScope ps(ar::CAT_CHUNK, reinterpret_cast<cudaStream_t>(stream), 0.0);
  return ar::launch_scatter_kept(y, B, W, reinterpret_cast<const long long*>(dst_offsets), lo, len, out, out_len, workspace,
                                 workspace_bytes, reinterpret_cast<cudaStream_t>(stream));
}

int ar_profile_enable(int on) { return ar::prof_enable(on); }
int ar_profile_read(double* ms, double* flops, long long* launches, int n) {
  AR_CHECK(ms && flops && launches && n >= 1 && n <= AR_PROFILE_CATEGORIES, AR_ERR_INVALID, "ar_profile_read: bad argument");
  return ar::prof_read(ms, flops, launches, n);
}
long long ar_launch_count(void) { return ar::prof_launch_count(); }

int ar_debug_conv1d(const float* x, const float* w_host, const float* bias_host, float* y, int B, int Cin, int Cout, int T, int k,
                    int dilation, int lrelu, int engine, void* stream) {
  return ar::debug_conv(x, w_host, bias_host, y, B, Cin, Cout, T, k, dilation, lrelu, engine, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
