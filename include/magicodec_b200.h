/* magicodec_b200.h — C ABI of the B200-native MagiCodec tokenization engine.
 *
 * This is the drop-in boundary of SURVEY.md §8(b).  The reference has no FFI of its own (it is
 * pure Python over third-party PyTorch modules); each entry point below names the reference
 * call it stands in for, file:line relative to /root/reference:
 *
 *   mc_create / mc_set_tensor / mc_finalize   load_magicodec_model(name, device)
 *                                             realtime_codec_agent/audio_tokenizer.py:27-28
 *   mc_encode                                 _magicodec_encode: pad_audio -> encoder ->
 *                                             quantizer.inference          audio_tokenizer.py:189-194
 *   mc_decode                                 _magicodec_decode: codebook_proj(codebook.weight) ->
 *                                             F.embedding -> decoder       audio_tokenizer.py:196-201
 *   mc_decode_latents                         model.decoder(z_q)           audio_tokenizer.py:200
 *   mc_vq_search                              model.quantizer.inference    audio_tokenizer.py:192
 *   mc_codebook                               quantizer.codebook_proj(quantizer.codebook.weight)
 *                                                                          audio_tokenizer.py:158,198
 *   mc_stream_set_emit / _push_codes_emit     RealtimeAgent.detokenize_output_chunk: detokenize_audio ->
 *                                             pad_or_trim -> normalize_audio_rms -> smooth_join
 *                                             realtime_agent_v2.py:556-579, utils/audio_utils.py:4-46
 *   mc_embed_distance                         F.embedding + vector_norm + mean of
 *                                             ExternalTTSDuplexAligner  external_tts_duplex_aligner.py:14-27
 *   mc_op_*                                   the library kernels underneath (cuDNN conv1d, cuBLAS /
 *                                             fused_dense_lib linears, flash-attn local attention,
 *                                             csrc/layer_norm, csrc/rotary; magicodec_build.sh:4-16)
 *
 * Conventions: every function returns 0 on success or a negative MC_ERR_* code and never throws
 * or aborts; mc_last_error() gives the message.  All tensor arguments are DEVICE pointers owned by
 * the caller (torch allocations on the host side); the library owns its handle, workspaces and
 * cached TMA descriptors only.  Calls are asynchronous with respect to `stream` and do not
 * synchronise (exception: a workspace that must grow synchronises the stream once).  A handle is
 * not thread-safe: one handle per thread/stream.  sm_100 only — mc_create fails with MC_ERR_ARCH
 * elsewhere; there is no CPU fallback.
 */
#ifndef MAGICODEC_B200_H_
#define MAGICODEC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MC_VERSION 100

enum {
  MC_OK = 0,
  MC_ERR_ARG = -1,      /* bad argument / shape / missing tensor */
  MC_ERR_ARCH = -2,     /* device is not sm_100 */
  MC_ERR_CUDA = -3,     /* CUDA runtime / driver error (message has the detail) */
  MC_ERR_STATE = -4,    /* call order (e.g. encode before finalize) */
  MC_ERR_NOMEM = -5
};

typedef struct mc_handle mc_handle;
typedef void* mc_stream_t; /* cudaStream_t */

#define MC_MAX_CONVS 8

typedef struct mc_spec {
  int32_t sample_rate;
  int32_t n_convs;                       /* encoder conv layers (decoder mirrors them)          */
  int32_t conv_channels[MC_MAX_CONVS];   /* output channels of each encoder conv; last = d_model */
  int32_t conv_strides[MC_MAX_CONVS];    /* kernel = 2*stride, causal                            */
  int32_t d_model, n_heads, ffn_dim;
  int32_t enc_layers, dec_layers;
  int32_t window_left, window_right;     /* attention keys j in [i-wl, i+wr]                     */
  float norm_eps;
  int32_t codebook_size, codebook_dim;
  int32_t max_positions;                 /* rows of the RoPE cos/sin tables                      */
} mc_spec;

int mc_version(void);
const char* mc_last_error(const mc_handle* h); /* h may be NULL: error of the last failed mc_create */

int mc_create(const mc_spec* spec, int device, mc_handle** out);
int mc_destroy(mc_handle* h);

/* Register one packed parameter (device pointer, kept by reference).  Names and layouts are listed
 * in DESIGN.md §"Packed weights"; mc_finalize checks that all of them are present. */
int mc_set_tensor(mc_handle* h, const char* name, const void* dev_ptr, int64_t numel);
int mc_finalize(mc_handle* h);

/* wav: fp32, B windows of T samples, window b starts at wav + b*ld (ld < T gives overlapping
 * windows: the chunked encode of audio_tokenizer.py:52-65 is ld = chunk samples, T = context).
 * T need not be a hop multiple (right zero padding = pad_audio).  F = ceil(T/hop).
 * keep_last_frames: 0 = all F frames, else only the last k frames of each window are quantised.
 * codes: int64 [B, Fk]; margin (optional): fp32 [B, Fk] = second-best minus best squared distance;
 * z_e (optional): fp32 [B, F, dq] encoder output before quantisation. */
int mc_encode(mc_handle* h, const float* wav, int64_t ld, int32_t B, int32_t T, int32_t keep_last_frames,
              int64_t* codes, float* margin, float* z_e, mc_stream_t stream);

/* codes: int64 [B, F].  keep_last_samples: 0 = all F*hop samples, else the last k (clamped).
 * wav: fp32 [B, Tk]. */
int mc_decode(mc_handle* h, const int64_t* codes, int32_t B, int32_t F, int32_t keep_last_samples, float* wav,
              mc_stream_t stream);
/* Same, entered with latents z_q fp32 [B, F, dq] (what F.embedding returns in the reference). */
int mc_decode_latents(mc_handle* h, const float* z_q, int32_t B, int32_t F, int32_t keep_last_samples,
                      float* wav, mc_stream_t stream);

/* Nearest neighbour of each z row (fp32 [M, dq]) in the projected codebook. */
int mc_vq_search(mc_handle* h, const float* z, int32_t M, int64_t* codes, float* margin, mc_stream_t stream);

/* Copies the cached projected codebook, fp32 [K, dq]. */
int mc_codebook(mc_handle* h, float* out, mc_stream_t stream);

/* GEMM with an RMSNorm folded into it (DESIGN.md §4): consumer — y = acc * rsqrt(sum(row_stats[row][0..n)) / K + eps) + bias
 * with A = bf16(x * gamma); producer (fp32 output modes) — additionally xb_out = bf16(x_new * xb_gamma) [M, N] and
 * stat_out [M, N/64] = per-row sums of x_new^2 per 64 columns.  mc_op_rowstats: the same pair from an fp32 matrix.
 * Stand in for csrc/layer_norm (dropout_add_rms_norm) + the linear that follows it (magicodec_build.sh:10-16). */
int mc_op_gemm_fused(mc_handle* h, const void* A, const void* W, const float* bias, int32_t M, int32_t N, int32_t K, int32_t act,
                     int32_t out_mode, void* out, const float* row_stats, int32_t row_stats_n, void* xb_out, const float* xb_gamma,
                     float* stat_out, int32_t rope_cols, int32_t rope_period, int32_t block_n, mc_stream_t stream);
int mc_op_rowstats(mc_handle* h, const float* x, const float* gamma, void* xb_out, float* stat_out, int32_t M, int32_t d,
                   mc_stream_t stream);

/* Debug: timeline of a pass (only in a library built with -DMC_TRACE; MC_ERR_STATE otherwise). */
int64_t mc_debug_trace(mc_handle* h, void* dev_buf, int64_t capacity_records);

/* ---- corpus ingest on the device: what _prep_audio_for_tokenization (audio_tokenizer.py:203-215: int16 -> float,
 * librosa.to_mono, librosa.resample) and the offline CLI's loader do on the host in the reference.
 * pcm: DEVICE pointer to interleaved frames [frames][channels] in `format`; out: planar fp32 [C_out, out_ld]
 * (C_out = 1 when mix_mono: mean over channels like np.mean(axis=0)). */
enum { MC_PCM_U8 = 0, MC_PCM_S16 = 1, MC_PCM_S24 = 2, MC_PCM_S32 = 3, MC_PCM_F32 = 4, MC_PCM_F64 = 5, MC_PCM_ULAW = 6, MC_PCM_ALAW = 7 };
int mc_op_pcm_to_f32(mc_handle* h, const void* pcm, int32_t format, int32_t big_endian, int32_t channels, int64_t frames,
                     int32_t mix_mono, float* out, int64_t out_ld, mc_stream_t stream);
/* Rational polyphase FIR resampler (scipy.signal.resample_poly semantics: taps already scaled by `up` and left-padded
 * for alignment, pre_remove = leading outputs dropped): in planar fp32 [C, in_ld] -> out planar fp32 [C, out_ld]. */
int mc_op_resample(mc_handle* h, const float* in, int64_t in_ld, int32_t channels, int64_t n_in, int32_t up, int32_t down,
                   const float* taps, int32_t n_taps, int64_t pre_remove, float* out, int64_t out_ld, int64_t n_out,
                   mc_stream_t stream);

/* Host-side FLAC decoder (no CUDA; libri-light ships as .flac and no audio library is installed offline — the
 * reference loads it through librosa/soundfile/libFLAC).  data: the whole file in HOST memory.  mc_flac_decode writes
 * interleaved [frames][channels] PCM: int16 for streams of <= 16 bits per sample (MC_PCM_S16), else int32 left-justified
 * (MC_PCM_S32); verifies every frame's CRC-8 / CRC-16 and the STREAMINFO sample count. */
int mc_flac_info(const uint8_t* data, int64_t n, int32_t* sample_rate, int32_t* channels, int32_t* bits, int64_t* total_samples);
int mc_flac_decode(const uint8_t* data, int64_t n, void* out, int64_t capacity_frames, int64_t* decoded);

/* ---- streaming sessions: the rolling context of tokenize_audio / detokenize_audio
 * (audio_tokenizer.py:72-74, 111-113) resident in HBM; the steady state is one CUDA-graph launch per
 * call.  chunk / codes / outputs are HOST pointers (staged through pinned memory); these calls
 * synchronise `stream` before returning because the caller consumes the result. */
typedef struct mc_stream mc_stream;
int mc_stream_create(mc_handle* h, int32_t channels, int32_t context_samples, int32_t max_chunk_samples, mc_stream** out);
int mc_stream_destroy(mc_stream* s);
int mc_stream_reset(mc_stream* s);                      /* AudioTokenizer.reset_context, :44-46 (also forgets the emit chain's previous chunk) */
int mc_stream_reset_part(mc_stream* s, int32_t audio, int32_t codes); /* drop only the audio and/or the code context */
/* Upload a context WITHOUT computing anything: the session's audio (code) context becomes the last
 * min(n, context) samples (frames) of the HOST array [C,n].  Re-seeds a session after a one-shot
 * tokenize / detokenize call changed the host-side context (audio_tokenizer.py:72-74, 111-113). */
int mc_stream_load_audio(mc_stream* s, const float* audio, int32_t n);
int mc_stream_load_codes(mc_stream* s, const int64_t* codes, int32_t n);
/* chunk fp32 [C,n]; codes_out int64 [C,keep_frames] (0 = every frame of the window). */
int mc_stream_push_audio(mc_stream* s, const float* chunk, int32_t n, int32_t keep_frames, int64_t* codes_out,
                         int32_t* frames_out, mc_stream_t stream);
/* codes int64 [C,n]; wav_out fp32 [C,keep_samples] (0 = the whole decoded window). */
int mc_stream_push_codes(mc_stream* s, const int64_t* codes, int32_t n, int32_t keep_samples, float* wav_out,
                         int32_t* samples_out, mc_stream_t stream);
int mc_stream_set_graphs(mc_stream* s, int32_t enabled); /* 0: direct launches (A/B timing, debugging) */

/* ---- session pool: many independent rolling contexts batched per call (SURVEY §8 f2).  tts_server.py:59,158
 * tokenizes every active stream chunk by chunk on one shared tokenizer, realtime_agent_resources.py:41-49 runs two
 * agents on one model; alone, each session is a batch-1 pass that streams every weight for 100 rows.  Sessions whose
 * contexts have the same length are pushed together as ONE B = n*channels launch.  Per session the semantics are those
 * of mc_stream_push_audio / mc_stream_push_codes.  slots: n distinct indices < max_sessions; chunks HOST fp32
 * [n][C][len] -> codes_out HOST int64 [n][C][keep]; codes HOST int64 [n][C][len] -> wav_out HOST fp32 [n][C][keep]. */
typedef struct mc_pool mc_pool;
int mc_pool_create(mc_handle* h, int32_t channels, int32_t context_samples, int32_t max_chunk_samples, int32_t max_sessions,
                   mc_pool** out);
int mc_pool_destroy(mc_pool* p);
int mc_pool_reset(mc_pool* p, int32_t slot, int32_t audio, int32_t codes);
int mc_pool_context_len(mc_pool* p, int32_t slot, int32_t* audio_len, int32_t* code_len);
int mc_pool_set_graphs(mc_pool* p, int32_t enabled);
int mc_pool_push_audio(mc_pool* p, const int32_t* slots, int32_t n, const float* chunks, int32_t len, int32_t keep_frames,
                       int64_t* codes_out, int32_t* frames_out, mc_stream_t stream);
int mc_pool_push_codes(mc_pool* p, const int32_t* slots, int32_t n, const int64_t* codes, int32_t len, int32_t keep_samples,
                       float* wav_out, int32_t* samples_out, mc_stream_t stream);

/* ---- post-decode emit chain of the agent loop (mono sessions), fused behind the decoder in the same
 * CUDA graph: detokenize_audio(codes, preroll = fade) -> pad_or_trim -> normalize_audio_rms (skipped when
 * target_rms <= 0) -> smooth_join with the previous chunk -> the chunk to emit.
 * set_emit: chunk_samples = agent chunk (n codes * hop), fade_samples = L of create_crossfade_ramps,
 * fade_in = HOST fp32 [L] rising ramp (fade_out is its mirror).  Resets the "previous chunk" state.
 * push_codes_emit: codes HOST int64 [n]; out HOST fp32 [2*chunk + L] = emitted chunk [chunk] ++ the L
 * cross-faded samples that replace the tail of the previous history chunk ++ the new history chunk
 * [chunk]; *had_prev = whether a previous chunk existed (0 on the first call after create/reset/set_emit). */
int mc_stream_set_emit(mc_stream* s, int32_t chunk_samples, int32_t fade_samples, float target_rms,
                       float silence_rms_threshold, const float* fade_in);
int mc_stream_push_codes_emit(mc_stream* s, const int64_t* codes, int32_t n, float* out, int32_t* had_prev,
                              mc_stream_t stream);
/* The same chain for the mono sessions of a pool, n of them in one launch (one CUDA graph: decoder + emit_chunk_pool_kernel).
 * set_emit: the parameters of mc_stream_set_emit, shared by every slot; every slot forgets its previous chunk.
 * push_codes_emit: codes HOST int64 [n][len] with len * hop == chunk; out HOST fp32 [n][2*chunk + L], item j laid out as
 * mc_stream_push_codes_emit's block.  Per slot the semantics are those of mc_stream_push_codes_emit; all slots of one
 * call must share the context length and *had_prev (first chunks and continuing chunks go in separate calls).
 * mc_pool_reset(slot, codes != 0) also forgets that slot's previous chunk. */
int mc_pool_set_emit(mc_pool* p, int32_t chunk_samples, int32_t fade_samples, float target_rms, float silence_rms_threshold,
                     const float* fade_in);
int mc_pool_push_codes_emit(mc_pool* p, const int32_t* slots, int32_t n, const int64_t* codes, int32_t len, float* out,
                            int32_t* had_prev, mc_stream_t stream);

/* ---- ragged pool calls: the same per-session semantics, but the sessions of one call may hold contexts of different
 * length (streams in their warm-up next to streams in steady state), in ONE launch.  Every window starts at row 0 of
 * the batch and reads zeros (codes: code 0) past its own end; the codec is causal for window_right == 0, so each
 * session's kept frames equal its lone pass (bit for bit with small_m_split_k = 0).  Equal lengths take the uniform
 * call (same results, same graphs); different lengths on a spec with window_right != 0 fail with MC_ERR_ARG.  Every
 * check runs before any work or state change.
 * push_audio_ragged: 1 <= keep_frames <= ceil(len / hop); codes_out HOST int64 [n][C][keep_frames], item j = the last
 *   keep_frames frames of its own window.
 * push_codes_ragged: 1 <= keep_samples <= ceil(capacity / hop) * hop; item j gets min(keep_samples, new_len_j * hop) samples,
 *   the last ones of its window, at the start of its wav_out row HOST fp32 [n][C][keep_samples] (zeros after them);
 *   samples_out HOST int32 [n] = that count per item.
 * push_codes_emit_ragged: mc_pool_push_codes_emit where first chunks may mix with continuing ones; the rules of
 *   mc_pool_push_codes_emit hold per item; had_prev HOST int32 [n].
 * graph_count: distinct graph keys seen and graphs captured (all push calls of the pool). */
int mc_pool_push_audio_ragged(mc_pool* p, const int32_t* slots, int32_t n, const float* chunks, int32_t len, int32_t keep_frames,
                              int64_t* codes_out, mc_stream_t stream);
int mc_pool_push_codes_ragged(mc_pool* p, const int32_t* slots, int32_t n, const int64_t* codes, int32_t len, int32_t keep_samples,
                              float* wav_out, int32_t* samples_out, mc_stream_t stream);
int mc_pool_push_codes_emit_ragged(mc_pool* p, const int32_t* slots, int32_t n, const int64_t* codes, int32_t len, float* out,
                                   int32_t* had_prev, mc_stream_t stream);
int mc_pool_graph_count(mc_pool* p, int32_t* keys, int32_t* captured);
/* The last n samples (1 <= n <= the slot's context length) of a slot's audio context -> HOST fp32 [C][n]. */
int mc_pool_read_audio(mc_pool* p, int32_t slot, float* out_host, int32_t n);

/* ---- live-stream ingest for pooled sessions whose clients send PCM at their own rate and sample format (48 / 44.1 kHz
 * int16 from WebRTC or a TTS engine): per chunk what AudioTokenizer._prep_audio_for_tokenization does on the host
 * (audio_tokenizer.py:203-215: int16 / 32768, the mean over channels for a mono codec, librosa.resample), done on the
 * device inside the push's graph.  Each chunk is resampled on its own with zero edges, as the reference does.
 * set_resampler: registers the polyphase plan of one input rate (the ResamplePlan of audio_io.resample_plan(sr_in, codec
 * rate): taps HOST fp32 [n_taps], already scaled by `up` and left-padded; pre_remove = leading outputs dropped).
 *   sr_in * up == codec rate * down; at most MC_POOL_MAX_RESAMPLERS rates per pool; registering a rate again replaces it.
 * reserve_pcm: fixes the pinned staging of the raw chunks at max_sessions chunks of max_in_channels x max_in_samples;
 *   afterwards a larger item fails with MC_ERR_ARG.  Without it the staging is sized at first use and grows when a call
 *   needs more.
 * push_pcm / push_pcm_ragged: mc_pool_push_audio / mc_pool_push_audio_ragged (same rules, same results) on the converted
 *   samples.  items HOST [n]: item j's chunk is planar [channels_in][ld] samples (MC_PCM_S16 or MC_PCM_F32, native byte
 *   order) at payload + offset_bytes, n_in per channel, at sample_rate (the codec's rate, or a registered one).  Every
 *   item must resample to `len` samples, ceil(n_in * up / down).  A pool with C > 1 channels needs channels_in == C; a
 *   mono pool takes 1..MC_POOL_MAX_MIX_CHANNELS channels and mixes them (fp32 mean, np.mean(axis=0) order).  Per item
 *   the staged samples are bit for bit mc_op_pcm_to_f32 followed by mc_op_resample on the same bytes.  Every check runs
 *   before any work or state change. */
#define MC_POOL_MAX_RESAMPLERS 8
#define MC_POOL_MAX_MIX_CHANNELS 8
typedef struct mc_pcm_chunk {
  int32_t format;        /* MC_PCM_S16 or MC_PCM_F32 */
  int32_t channels_in;
  int32_t n_in;          /* samples per channel */
  int32_t sample_rate;
  int64_t offset_bytes;  /* of channel 0 in payload */
  int64_t ld;            /* samples from one channel's row to the next */
} mc_pcm_chunk;
int mc_pool_set_resampler(mc_pool* p, int32_t sr_in, int32_t up, int32_t down, const float* taps, int32_t n_taps, int64_t pre_remove);
int mc_pool_reserve_pcm(mc_pool* p, int32_t max_in_samples, int32_t max_in_channels);
int mc_pool_push_pcm(mc_pool* p, const int32_t* slots, int32_t n, const mc_pcm_chunk* items, const void* payload, int32_t len,
                     int32_t keep_frames, int64_t* codes_out, int32_t* frames_out, mc_stream_t stream);
int mc_pool_push_pcm_ragged(mc_pool* p, const int32_t* slots, int32_t n, const mc_pcm_chunk* items, const void* payload, int32_t len,
                            int32_t keep_frames, int64_t* codes_out, mc_stream_t stream);

/* ids DEVICE int64 [rows, n] (LM token ids; code = id - vocab_start, clamped to the codebook).
 * dist_out DEVICE fp32 [rows] (optional) = mean_j ||E[code_j] - ref||_2, ref DEVICE fp32 [dq] (NULL = 0);
 * mean_out DEVICE fp32 [rows, dq] (optional) = mean_j E[code_j], E = the cached projected codebook. */
int mc_embed_distance(mc_handle* h, const int64_t* ids, int32_t rows, int32_t n, int64_t vocab_start, const float* ref,
                      float* dist_out, float* mean_out, mc_stream_t stream);

/* Number of kernels launched by this handle since creation (bench.py's gpu_launches). */
int64_t mc_launch_count(const mc_handle* h);
/* Device timing by kernel class (0 GEMM, 1 attention, 2 VQ search, 3 HBM-bound elementwise): between
 * begin and end every launch is bracketed by a CUDA event pair on its stream; end synchronises on
 * those events and returns, per class, the summed milliseconds, algorithmic FLOPs and bytes, and
 * the launch count.  Used by bench.py for the roofline object; off by default. */
int mc_profile_begin(mc_handle* h);
int mc_profile_end(mc_handle* h, double* ms, double* flops, double* bytes, int64_t* launches, int32_t n_classes);
/* Engine options (all default to 1): "shared_stem" — overlapping hop-aligned windows of one mc_encode call share a
 * single pass of the convolution stack (bit-identical results; 0 recomputes it per window, for A/B tests);
 * "gemm_pair" — cta_group::2 GEMM where the shape allows; "fast_epilogue" — its mode-specialised epilogues
 * (bit-identical to the generic one); "attn_p_tmem" — attention keeps P in tensor memory (0: the shared-memory-P
 * kernel, bit-identical); "pdl" — programmatic dependent launch between the kernels of a pass; "exact_cut" — the
 * transformer layers drop rows no kept output depends on at the exact row (0: only in steps of 16 frames, the earlier
 * plan; bit-identical). */
int mc_set_option(mc_handle* h, const char* key, int32_t value);
/* impl: 0 = tensor-core kernels (default), 1 = SIMT cross-check kernels for attention / VQ; attention also
 * 2 = one-item-per-CTA tcgen05 kernel, 3 = two-slot persistent kernel without staged loads (A/B timing);
 * attention_impl bit 2 forces the single-CTA GEMM. */
int mc_set_debug_impl(mc_handle* h, int32_t attention_impl, int32_t vq_impl);

/* ---- operator level (each is one kernel launch; used by the parity tests and profiling) ---- */

/* out[M,N] = epilogue(A * W^T).  A bf16 viewed as [a_rows, a_k_wrap] row blocks, K = multiple of
 * a_k_wrap (see gemm_sm100.cuh); W bf16 [N,K]; bias fp32 [N] or NULL; act 0/1 (tanh-GELU);
 * out_mode 0 bf16 / 1 fp32 / 2 fp32 residual (out += result); rope_period > 0 applies RoPE from the
 * handle's tables to columns [0, rope_cols).  grp_in > 0 groups the M rows (grp_in per batch item, the
 * first grp_valid of them stored) and writes row r of group g at out + g*grp_stride + grp_off + r*ldo
 * (elements) — the implicit-GEMM convolutions; grp_in = 0 is a plain GEMM. */
int mc_op_gemm(mc_handle* h, const void* A, int64_t a_rows, int32_t a_k_wrap, const void* W, const float* bias,
               int32_t M, int32_t N, int32_t K, int32_t act, int32_t out_mode, void* out, int64_t ldo,
               int32_t grp_in, int32_t grp_valid, int64_t grp_stride, int64_t grp_off, int32_t rope_cols,
               int32_t rope_period, int32_t block_n, mc_stream_t stream);
int mc_op_rmsnorm(mc_handle* h, const float* x, const float* gamma, void* out_bf16, int32_t M, int32_t d,
                  mc_stream_t stream);
/* qkv bf16 [B*F, 3*d] (RoPE applied) -> out bf16 [B*out_rows, d]: the last out_rows queries of every window.
 * phase (0 .. 15): the window is the tail of a longer one, (F_full - F) mod 16 frames past a 16-frame boundary; the
 * tensor-core kernels then sum keys in the same groups as the full window, bit for bit.  0 for a whole window. */
int mc_op_attention(mc_handle* h, const void* qkv, void* out, int32_t B, int32_t F, int32_t out_rows, int32_t phase,
                    int32_t impl, mc_stream_t stream);

/* The two kernels behind mc_stream_push_codes_emit / mc_embed_distance on caller-supplied DEVICE buffers
 * (the golden-vector replays of tests/test_gpu_post.py): wav [n_have], fade_in / prev_tail [fade] (prev_tail is
 * updated in place), out [2*chunk + fade]; table fp32 [K,16]. */
int mc_op_emit_chunk(mc_handle* h, const float* wav, int32_t n_have, int32_t chunk, int32_t fade, int32_t has_prev,
                     float target_rms, float silence_rms_threshold, const float* fade_in, float* prev_tail, float* out,
                     mc_stream_t stream);
int mc_op_embed_distance(mc_handle* h, const float* table, int32_t K, const int64_t* ids, int32_t rows, int32_t n,
                         int64_t vocab_start, const float* ref, float* dist_out, float* mean_out, mc_stream_t stream);

/* ---- offline corpus decode (the way back from a directory of codes; python -m rca_b200_loader codes_to_audio).
 * mc_render_chunks: the agent's output chain (OutputChunkEmitter; RealtimeAgent.detokenize_output_chunk,
 * realtime_agent_v2.py:556-579: pad_or_trim -> normalize_audio_rms (skipped when target_rms <= 0) -> smooth_join) for
 * EVERY chunk of one mono stream in one launch; the result equals mc_op_emit_chunk run chunk by chunk, bit for bit.
 * windows DEVICE fp32 [n_chunks, ld]: row 0 = the first chunk's decoded samples, rows i >= 1 = fade preroll ++ chunk;
 * the last row holds last_len new samples (a ragged last chunk).  fade_in DEVICE fp32 [fade] rising ramp.
 * out DEVICE fp32 [(n_chunks-1)*chunk + last_len] = np.concatenate(audio_history_ch1) cut to the real samples.
 * Needs 0 < fade <= chunk, 0 < last_len <= chunk, ld >= chunk + fade. */
int mc_render_chunks(mc_handle* h, const float* windows, int64_t ld, int32_t n_chunks, int32_t chunk, int32_t fade,
                     int32_t last_len, float target_rms, float silence_rms_threshold, const float* fade_in, float* out,
                     mc_stream_t stream);
/* The CLI's writer (the reference's consumers write wav files through soundfile): planar fp32 [channels, in_ld] ->
 * interleaved [frames][channels] as MC_PCM_S16 (clamp(rint(x * 32768), -32768, 32767), NaN -> 0: the inverse of the
 * / 32768 of _prep_audio_for_tokenization, audio_tokenizer.py:203-215) or MC_PCM_F32.  in is a DEVICE pointer; out may
 * be DEVICE or PINNED HOST memory. */
int mc_op_f32_to_pcm(mc_handle* h, const float* in, int64_t in_ld, int32_t channels, int64_t frames, int32_t format, void* out,
                     mc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MAGICODEC_B200_H_ */
