/*
 * audiorestore.h -- C-ABI of libaudiorestore_sm100.so (B200 / sm_100a).
 *
 * The reference (JonathanBedrava/ml-audio-restoration) is pure Python/PyTorch and has no FFI
 * of its own; these entry points are what a binding for its inference hot path would bind.
 * Each one names the reference interface it replaces (file:line under the reference root).
 *
 * Conventions
 *   - every function returns 0 on success, a non-zero AR_ERR_* code otherwise;
 *     ar_last_error() returns a thread-local human-readable message (the Python shim turns
 *     it into RuntimeError/ValueError, preserving the reference's exception convention).
 *   - all pointers named x/y/audio/chunks/out/workspace are DEVICE pointers unless the
 *     function name ends in _host; the caller owns them.  Handles own the packed weights.
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no entry point
 *     synchronises the device except the *_create functions (weight upload), the diagnostic
 *     ar_model_audit_* pair and ar_debug_conv1d.
 *   - a process may drive several GPUs: handles belong to the device they were created on, calls
 *     are made with that device current (the Python shim does), kernel attributes are set per device.
 *   - tensors are fp32, contiguous, in the reference's layout: audio batches are
 *     [B,1,T], stereo outputs [B,2,T] (denoiser.py:93, super_resolution.py:69,
 *     stereo_separator.py:88).
 *   - there is no CPU fallback: on a machine without an sm_100 device *_create fails.
 */
#ifndef AUDIORESTORE_H_
#define AUDIORESTORE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AR_OK 0
#define AR_ERR_INVALID 1   /* bad argument / shape (reference: RuntimeError from ATen)      */
#define AR_ERR_WEIGHTS 2   /* missing / mis-shaped state_dict entry (load_state_dict strict) */
#define AR_ERR_CUDA 3      /* CUDA runtime failure                                           */
#define AR_ERR_WORKSPACE 4 /* workspace too small                                            */

#define AR_MODEL_DENOISER 0  /* AudioDenoiser()                       denoiser.py:6          */
#define AR_MODEL_SUPER_RES 1 /* AudioSuperResolution(upscale_factor=2) super_resolution.py:6 */
#define AR_MODEL_STEREO 2    /* StereoSeparator(32, 64, 1)            stereo_separator.py:5  */

#define AR_ENGINE_UMMA 0 /* tcgen05 implicit-GEMM conv engines (product path)                */
#define AR_ENGINE_SIMT 1 /* CUDA-core fp32 conv engine (debug cross-check only)              */

typedef struct ar_model_s* ar_model_t;
typedef struct ar_chain_s* ar_chain_t;

/* One state_dict entry: HOST pointer to contiguous fp32 data (int64 num_batches_tracked
 * entries are not passed; eval-mode BatchNorm ignores them, SURVEY.md App. B.4). */
typedef struct {
  const char* name;  /* exact reference key, e.g. "encoder.0.0.weight" (App. C)            */
  const float* data; /* host fp32                                                           */
  int ndim;
  int64_t shape[4];
} ar_tensor_t;

const char* ar_last_error(void);
int ar_version(void);

/* Select the conv engine used by subsequently created models (default AR_ENGINE_UMMA). */
int ar_set_conv_engine(int engine);

/* Fused multi-layer launches (the StereoSeparator's dilated block conv k3 -> conv k1 [-> LSTM input projection],
 * stereo_separator.py:49-64,104-106, and the U-Net's / residual blocks' conv k3 -> conv k3 pairs, denoiser.py:51-60,
 * super_resolution.py:104-122, as one kernel whose intermediates stay in shared memory) for subsequently created
 * models: 0 = layer by layer, 1 (default) = every chain that fits; anything else is AR_ERR_INVALID.  Cross-check knob:
 * both settings compute the same fp16-rounded intermediates. */
int ar_set_fusion(int on);

/* Replaces: model construction + torch.load + load_state_dict(strict) + .to(device) + .eval()
 * (inference.py:51-55, 66-70, 85-89).  Folds eval-mode BatchNorm into the conv weights,
 * rounds tensor-core operands to fp16 (the 11-bit significand TF32 would keep), packs into the kernels' layouts, uploads.
 * An optional entry "<bn>.eps" (shape [1]) overrides nn.BatchNorm1d's default eps = 1e-5 for that layer.
 * AR_ERR_WEIGHTS: missing / mis-shaped entry, or a BatchNorm-folded weight outside the fp16 operand range
 * (|w| > 65504, not finite, or a whole layer below 6.1e-5) -- refused, never clamped silently. */
int ar_model_create(int kind, const ar_tensor_t* tensors, int n_tensors, int device, ar_model_t* out);
void ar_model_destroy(ar_model_t m);
int ar_model_kind(ar_model_t m);

/* Bytes of device scratch ar_model_forward needs for a [B,1,T] batch. */
int ar_model_workspace_bytes(ar_model_t m, int B, int T, size_t* bytes);

/* Replaces nn.Module.forward under eval()/no_grad():
 *   denoiser  : x[B,1,T] -> y[B,1,T]    (denoiser.py:88-144; T >= 8 else AR_ERR_INVALID)
 *   super-res : x[B,1,T] -> y[B,1,2T]   (super_resolution.py:66-101)
 *   stereo    : x[B,1,T] -> y[B,2,T]    (stereo_separator.py:85-122; LSTM state starts at 0) */
int ar_model_forward(ar_model_t m, const float* x, float* y, int B, int T,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Dynamic-range audit of a checkpoint (diagnostic; INTEGRATION.md "dynamic range").  Activations between layers are
 * stored in fp16 and SATURATE at +-65504; random-init and BatchNorm-calibrated checkpoints stay orders of magnitude below,
 * but nothing in the state_dict ABI guarantees it.  While the audit is on, forwards of this model run layer by layer
 * (fused launches off) and record max |activation| of every fp16 tensor they write; ar_model_audit_read synchronises the
 * device and returns them in launch order (n_layers <= AR_AUDIT_MAX_LAYERS; names via ar_model_audit_name).  A maximum
 * of 65504 means that layer clipped.  Not re-entrant: one audited forward at a time per model. */
#define AR_AUDIT_MAX_LAYERS 64
int ar_model_audit_enable(ar_model_t m, int on);
int ar_model_audit_read(ar_model_t m, float* max_abs, int cap, int* n_layers);
const char* ar_model_audit_name(ar_model_t m, int i);
/* Test hook on the audit path: while the audit is on, every forward that writes the audited tensor `name` also copies the
 * channel window it wrote into the device buffer y as plain fp32 [B][channels][T] (rows [0,T) only).  Several names may be
 * armed at once; arming a name again replaces its buffer; a NULL name disarms all.  A window of more than cap_floats
 * values makes that forward return AR_ERR_INVALID before the copy is launched.  Forwards with the audit off ignore taps. */
int ar_model_audit_tap(ar_model_t m, const char* name, float* y, int64_t cap_floats);

/* Stereo forward with explicit LSTM carry (whole-file-exact mode, SURVEY.md 8 n2):
 * state_in/state_out are [B,2,64] (h then c) device buffers; either may be NULL. */
int ar_stereo_forward_state(ar_model_t m, const float* x, float* y, int B, int T,
                            const float* state_in, float* state_out,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Stereo forward on a WINDOW of a longer signal (whole-file-exact chunked mode): x[B,1,T] is a segment that carries conv
 * halos on both sides.  The encoder and the decoders run over all T samples; the LSTM scan covers steps [lstm_start, T)
 * only, starting from state_in (NULL = zeros; hidden states of earlier steps are zero), and state_out receives (h, c)
 * after step state_pos - 1 (lstm_start < state_pos <= T) -- the state the NEXT segment's scan starts from, taken where
 * this segment's LSTM inputs are still exact.  lstm_start and state_pos are multiples of 8 (state_pos may equal T).
 * Chaining segments this way reproduces the single scan of stereo_separator.py:106-107 over the whole file. */
int ar_stereo_forward_window(ar_model_t m, const float* x, float* y, int B, int T, int lstm_start, int state_pos,
                             const float* state_in, float* state_out,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ar_stereo_forward_window for B windows that hand their state on at different steps (lockstep whole-file-exact mode over
 * many files): state_pos is a HOST array of B entries, lstm_start < state_pos[b] <= T, any integers; state_out[b] receives
 * (h, c) after step state_pos[b] - 1 while the scan of item b runs on to T in the same launch.  The array is checked on the
 * host and uploaded into the workspace (counted by ar_model_workspace_bytes) on `stream`; no host synchronisation.
 * Outputs and states equal those of ar_stereo_forward_window on the same batch with state_pos = state_pos[b]. */
int ar_stereo_forward_window_multi(ar_model_t m, const float* x, float* y, int B, int T, int lstm_start, const int* state_pos,
                                   const float* state_in, float* state_out,
                                   void* workspace, size_t workspace_bytes, void* stream);

/* Window gather / kept-range scatter (lockstep whole-file-exact mode, one launch per direction for all files):
 *   ar_gather_windows : dst[b][0][0..W) = src[offsets[b] .. offsets[b] + W)             (0 <= offsets[b] <= src_len - W)
 *   ar_scatter_kept   : out[dst_offsets[2b + c] + j] = y[b][c][lo[b] + j], j < len[b], c = 0, 1  (y is [B,2,W];
 *                       0 <= lo[b], lo[b] + len[b] <= W, dst_offsets[2b + c] + len[b] <= out_len)
 * Offsets and ranges are HOST arrays, checked on the host and uploaded into `workspace` (>= B * AR_WINDOW_IO_BYTES_PER_ITEM
 * device bytes, not reused by the caller before the launch has run) on `stream`; no host synchronisation. */
#define AR_WINDOW_IO_BYTES_PER_ITEM 24
int ar_gather_windows(const float* src, int64_t src_len, const int64_t* offsets, int B, int W, float* dst,
                      void* workspace, size_t workspace_bytes, void* stream);
int ar_scatter_kept(const float* y, int B, int W, const int64_t* dst_offsets, const int* lo, const int* len, float* out,
                    int64_t out_len, void* workspace, size_t workspace_bytes, void* stream);

/* denoise -> (super-res) -> stereo on a batch of equal-length chunks
 * (the three model applications of inference.py:59-61,73-75,93-95).  sr may be NULL
 * (enable_super_resolution=False): y is [B,2,T] instead of [B,2,2T].
 * Any B is one call.  Up to 8 chunks per SM the three forwards run on the whole batch; beyond that (16 per SM fills
 * the chip with ONE launch of the LSTM scan kernel) the convs run on sub-batches of 8 per SM around a single scan over
 * all B sequences, which then computes the LSTM input projection itself -- ar_chain_workspace_bytes accounts for it
 * (about 68 MB per chunk up to 8 per SM, 54 MB per chunk at 16 per SM: 128 GB for 2368 two-second chunks). */
int ar_chain_create(ar_model_t denoiser, ar_model_t sr, ar_model_t stereo, ar_chain_t* out);
void ar_chain_destroy(ar_chain_t c);
int ar_chain_workspace_bytes(ar_chain_t c, int B, int T, size_t* bytes);
int ar_chain_forward(ar_chain_t c, const float* x, float* y, int B, int T,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Replaces normalize_audio (audio_processing.py:58-87) without its two host syncs:
 * in-place RMS -> target_db over all n elements, then peak-limit to 1.0; rms==0 leaves the
 * data untouched.  scratch: >= AR_NORMALIZE_SCRATCH_BYTES of device memory. */
#define AR_NORMALIZE_SCRATCH_BYTES 16384
int ar_normalize(float* audio, int64_t n, float target_db, void* scratch, void* stream);

/* Front end of load_audio (audio_processing.py:10-42) on the device:
 *   ar_pcm16_to_float : interleaved PCM16 frames [n][channels] -> planar fp32 [channels][n] (x / 32768, as
 *                       soundfile's float32 read at :24)
 *   ar_resample_mono  : planar fp32 [channels][n] -> mono fp32 [n_out]: torch.mean(dim=0) (:33) fused with
 *                       torchaudio.transforms.Resample(orig_sr, new_sr) (:38; sinc_interp_hann, lowpass_filter_width 6,
 *                       rolloff 0.99 polyphase FIR).  n_out must be ar_resample_length() = ceil(new * n / orig)
 *                       (== n when the rates match: then only the mono mix is applied). */
int ar_resample_length(int64_t n, int orig_sr, int new_sr, int64_t* n_out);
int ar_resample_mono(const float* x, int channels, int64_t n, int orig_sr, int new_sr, float* y, int64_t n_out, void* stream);
int ar_pcm16_to_float(const int16_t* pcm, int channels, int64_t n, float* y, void* stream);
/*   ar_pcm_to_float   : the same for every sample encoding a RIFF/WAVE `data` chunk carries -- interleaved little-endian
 *                       frames [n][channels] of `format` -> planar fp32 [channels][n], scaled as soundfile's float32
 *                       read (:24) scales them: unsigned 8-bit (x - 128) / 128, signed 16 / 24 (packed) / 32-bit
 *                       x / 2^(bits-1), IEEE float32 as is, float64 rounded to nearest.  `raw` must be aligned to the
 *                       sample size (the packed 24-bit format to 1). */
#define AR_PCM_U8 1
#define AR_PCM_S16 2
#define AR_PCM_S24 3
#define AR_PCM_S32 4
#define AR_PCM_F32 5
#define AR_PCM_F64 6
int ar_pcm_to_float(const void* raw, int format, int channels, int64_t n, float* y, void* stream);

/* FLAC input for the same front end: sf.read of a .flac file (audio_processing.py:24), decoded on the device (RFC 9639).
 *   ar_flac_workspace_bytes : device scratch ar_flac_decode needs for `nbytes` bytes of frame data
 *   ar_flac_decode          : frames[nbytes] = the frame section of one stream (DEVICE bytes after the metadata blocks);
 *                             channels / bps / sample_rate / min_block / max_block / total_samples are the STREAMINFO
 *                             fields (total_samples 0 = unknown) -> planar fp32 y[channels][n] (row stride n),
 *                             x / 2^(bps-1) as soundfile's float32 read scales it (bit-exact for bps <= 24; 32-bit through
 *                             __int2float_rn, as AR_PCM_S32).  *n_out receives the samples per channel; y == NULL only
 *                             counts them (for total_samples 0).  Frames are found by a frame-parallel index of sync codes,
 *                             chained from byte 0 and decoded one thread per frame.  Synchronises `stream` to read the
 *                             frame table back (a loader that runs once per file).  A malformed stream -- CRC-8 / CRC-16
 *                             mismatch, reserved code, truncation, a change of rate / depth / channels mid-stream, frames
 *                             that disagree with total_samples -- returns AR_ERR_INVALID with a message naming the frame
 *                             index and byte offset in `frames`.  MD5 is not checked (libFLAC's default too). */
int ar_flac_workspace_bytes(int64_t nbytes, size_t* bytes);
int ar_flac_decode(const uint8_t* frames, int64_t nbytes, int channels, int bps, int sample_rate, int min_block, int max_block,
                   int64_t total_samples, float* y, int64_t n, int64_t* n_out, void* workspace, size_t workspace_bytes,
                   void* stream);

/* FLAC output: torchaudio.save of a .flac path (audio_processing.py:45-55), encoded on the device (RFC 9639).
 *   ar_flac_encode_workspace_bytes : device scratch (*workspace) and frame-output bytes (*out_capacity) ar_flac_encode needs
 *                             for `channels` x `n` samples at `block_size` and `bps`; AR_ERR_INVALID for arguments
 *                             ar_flac_encode rejects
 *   ar_flac_encode          : x = planar fp32 [channels][n] (DEVICE), channels 1..8, bps 16 or 24, sample_rate 1..655350,
 *                             block_size 16..4608 -> frames_out[out_capacity] (DEVICE) = the frame section of the stream
 *                             (the caller writes `fLaC` and STREAMINFO in front: min = max block = block_size) and
 *                             pcm_le_out (DEVICE, n * channels * bps / 8 bytes) = the interleaved little-endian samples
 *                             the STREAMINFO MD5 is taken over.  Samples are rint_even(clamp(x, -1, 1) * (2^(bps-1) - 1))
 *                             (fp32 multiply; NaN -> 0), as the pcm16 WAV writer rounds.  Fixed blocking (frame numbers,
 *                             short last frame); per channel the fewest exact bits of CONSTANT, FIXED orders 0..4 (Rice /
 *                             Rice2 and partition order searched exactly) and VERBATIM, with wasted bits; for two
 *                             channels the cheapest of independent / left-side / side-right / mid-side.  The output is
 *                             byte-identical to tests/flac_encode_ref.py::encode_search.  *frame_bytes_total, *min_frame,
 *                             *max_frame receive the bytes of the frame section and of its smallest and largest frame.
 *                             Synchronises `stream` once to read them.  A frame that did not write exactly the bits it
 *                             was sized for returns AR_ERR_INVALID naming the frame. */
int ar_flac_encode_workspace_bytes(int channels, int64_t n, int block_size, int bps, size_t* workspace, size_t* out_capacity);
int ar_flac_encode(const float* x, int channels, int64_t n, int bps, int sample_rate, int block_size, uint8_t* frames_out,
                   size_t out_capacity, uint8_t* pcm_le_out, int64_t* frame_bytes_total, int* min_frame, int* max_frame,
                   void* workspace, size_t workspace_bytes, void* stream);

/* Synthetic 78 rpm degradation generator (simulate_vinyl_artifacts, audio_processing.py:122-226; SURVEY.md 8f n4).
 * The random draws (np.random levels / pop plan, torch.randn noise tensors) stay with the caller; these entry points
 * are the deterministic arithmetic, rows = channels (or any batch of equal-length rows), all device fp32 [rows][n]:
 *   ar_butter       : scipy.signal.butter(order, wn, 'low' | 'high') as used at :196,208,220 -- HOST function,
 *                     b / a receive order+1 float64 coefficients, order <= 4
 *   ar_vinyl_mix    : y = audio + surface_noise * surface_level (:152-153), then every pop of `pops` (DEVICE array,
 *                     draw order) added to all rows (:157-188): float64 `amp_signed * exp(-k / tau)` plus, when
 *                     has_resonance, `0.3 * sin(omega * k / sample_rate) * decay * amp * 0.2`, rounded to float32
 *   ar_filtfilt     : y = float32(scipy.signal.filtfilt(b, a, row)) of row = scale * x (+ add1) (+ add2) (float32 sums;
 *                     add1 / add2 may be NULL): odd extension by 3*(order+1) samples, lfilter_zi initial state, forward
 *                     and backward float64 passes (:197-199, 209-211, 221-223).  n <= 3*(order+1) -> AR_ERR_INVALID
 *                     (scipy: ValueError).  y may alias x / add1 / add2.
 *   ar_vinyl_sum    : y = x0 (+ x1) (+ x2), float32 left to right (the `+ crackle`, `+ rumble` of :200,213 when no
 *                     roll-off filter follows) */
typedef struct {
  int64_t loc;           /* first sample                                                    */
  int32_t length;        /* min(int(sample_rate * decay_time), n - loc)                     */
  int32_t has_resonance; /* length > 10                                                     */
  double amp_signed;     /* amp * polarity                                                  */
  double amp;
  double tau;            /* sample_rate * decay_time * 0.3                                  */
  double omega;          /* 2 * pi * resonance_freq                                         */
} ar_pop_t;
int ar_butter(int order, double wn, int highpass, double* b, double* a);
int ar_vinyl_mix(const float* audio, const float* surface_noise, float surface_level, const ar_pop_t* pops, int n_pops,
                 int sample_rate, float* y, int rows, int64_t n, void* stream);
int ar_vinyl_sum(const float* x0, const float* x1, const float* x2, float* y, int64_t count, void* stream);
int ar_filtfilt_workspace_bytes(int rows, int64_t n, int order, size_t* bytes);
int ar_filtfilt(const float* x, float scale, const float* add1, const float* add2, float* y, int rows, int64_t n,
                const double* b, const double* a, int order, void* workspace, size_t workspace_bytes, void* stream);

/* Chunk / stitch (vocabulary of chunk_audio, audio_processing.py:229-253; tail zero-pad of
 * trainer.py:656-665).  hop = chunk_size - overlap, overlap <= chunk_size/2.
 *   ar_num_chunks     : chunks needed for n samples
 *   ar_split_chunks   : audio[n] -> chunks[n_chunks,1,chunk_size] for chunk indices
 *                       [first, first+count)
 *   ar_overlap_add    : y[n_chunks,C,rate*chunk_size] -> out[C, rate*n] with linear
 *                       cross-fades over rate*overlap samples (gather form, deterministic) */
int ar_num_chunks(int64_t n, int chunk_size, int overlap, int* n_chunks);
int ar_split_chunks(const float* audio, int64_t n, float* chunks, int first, int count,
                    int chunk_size, int overlap, void* stream);
int ar_overlap_add(const float* y, float* out, int64_t n, int n_chunks, int channels,
                   int chunk_size, int overlap, int rate, void* stream);

/* Measurement hooks (bench.py): kernels launched so far by this library, and -- while enabled --
 * CUDA-event timing of every launch on its own stream, summed per category
 * (0 conv engine, 1 LSTM recurrence, 2 stems, 3 tails, 4 normalize, 5 split/overlap-add).
 * ar_profile_read synchronises on the recorded events, returns the sums since the last read
 * (ms, algorithmic FLOPs, launch counts; arrays of n <= AR_PROFILE_CATEGORIES) and clears them. */
#define AR_PROFILE_CATEGORIES 6
int ar_profile_enable(int on);
int ar_profile_read(double* ms, double* flops, long long* launches, int n);
long long ar_launch_count(void);

/* Debug / test hook: one conv layer on channel-blocked activations through the selected
 * engine; lets tests compare the tcgen05 engine with the SIMT one layer by layer.
 * x: [B,Cin,T] plain fp32, w: [Cout,Cin,k] host fp32, bias: [Cout] host fp32,
 * y: [B,Cout,T] plain fp32 (device).  */
int ar_debug_conv1d(const float* x, const float* w_host, const float* bias_host, float* y,
                    int B, int Cin, int Cout, int T, int k, int dilation, int lrelu,
                    int engine, void* stream);

/* Debug / tuning hook: while dev_buf != NULL, every fused-chain launch records clock64() timestamps of the
 * pipeline events of its first 64 tile pairs (cluster 0) into slot (k mod 8) of dev_buf[8][64*16] (device int64),
 * k = launches since this call. */
int ar_debug_chain_trace(long long* dev_buf);

#ifdef __cplusplus
}
#endif
#endif /* AUDIORESTORE_H_ */
