// Rows f3 / f4 of SURVEY §8: the steps that sit directly behind the decoder in the agent loop.
//
//   emit_chunk_kernel      pad_or_trim -> normalize_audio_rms -> smooth_join crossfade -> the chunk
//                          the agent emits (realtime_agent_v2.py:556-579, utils/audio_utils.py:4-46)
//   emit_chunk_pool_kernel the same chain for every session of a session-pool batch in one launch
//   emit_chunks_kernel     the same chain for every chunk of a stream in one launch (offline render)
//   embed_distance_kernel  F.embedding of code ids + distance to a reference embedding + mean
//                          (external_tts_duplex_aligner.py:14-27)
//
// Both touch a few KB: one CTA, fixed-order reductions (bit-reproducible run to run), fp64 sums so
// the statistics are closer to the exact value than numpy's fp32 pairwise sums are.
#pragma once
#include "engine_common.cuh"

namespace mc {

constexpr int POST_THREADS = 256;

// Sum over the block, identical order every launch: per-thread serial partials -> fixed shuffle
// tree -> fixed smem tree.  Result valid in every thread.
__device__ __forceinline__ double block_sum_f64(double v, double* scratch /*[POST_THREADS/32 + 1]*/) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (blockDim.x >> 5); ++w) t += scratch[w];
    scratch[POST_THREADS / 32] = t;
  }
  __syncthreads();
  return scratch[POST_THREADS / 32];
}

// One channel (the agent's output channel is mono; pad_or_trim rejects anything else).
//   wav      [n_have]  decoder output tail: `n_pre` preroll samples then the new chunk
//   prev_tail[L]       last L samples of the previous history chunk (state, updated in place)
//   fade_in  [L]       rising ramp; fade_out is its mirror image (create_crossfade_ramps, :19-23)
//   out      [chunk + L + chunk]:
//       [0, chunk)                emitted chunk
//       [chunk, chunk + L)        cross-faded samples that replace the tail of the previous history chunk
//       [chunk + L, 2*chunk + L)  the new history chunk
// has_prev = 0 (first chunk of a session): n_have = chunk (no preroll was available); the chunk is
// emitted delayed by L behind L zeros and becomes the history as is.
__device__ __forceinline__ void emit_chunk_body(const float* __restrict__ wav, int n_have, int chunk, int L, int has_prev,
                                                float target_rms, float silence_thr, const float* __restrict__ fade_in,
                                                float* __restrict__ prev_tail, float* __restrict__ out, double* scratch) {
  const int want = has_prev ? chunk + L : chunk;       // pad_or_trim target (right pad with zeros / trim)
  const int n = min(n_have, want);
  float scale = 1.0f;
  if (target_rms > 0.0f) {
    double ss = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const double v = static_cast<double>(wav[i]);
      ss += v * v;
    }
    ss = block_sum_f64(ss, scratch);
    const float rms = sqrtf(static_cast<float>(ss / static_cast<double>(want)));
    if (rms >= silence_thr) scale = target_rms / rms;
  }
  auto x = [&](int i) -> float { return i < n ? __fmul_rn(wav[i], scale) : 0.0f; };   // padded, normalised chunk
  float* emit = out;
  float* fix = out + chunk;
  float* hist = out + chunk + L;
  if (has_prev) {
    for (int i = threadIdx.x; i < chunk; i += blockDim.x) {
      float e;
      if (i < L) {
        // separate roundings like numpy's tail1 * fade_out + head2 * fade_in (no FMA contraction)
        e = __fadd_rn(__fmul_rn(prev_tail[i], fade_in[L - 1 - i]), __fmul_rn(x(i), fade_in[i]));
        fix[i] = e;
      } else {
        e = x(i);
      }
      emit[i] = e;
      hist[i] = x(L + i);
    }
    __syncthreads();   // every read of prev_tail above is done
    for (int i = threadIdx.x; i < L; i += blockDim.x) prev_tail[i] = x(chunk + i);
  } else {
    for (int i = threadIdx.x; i < chunk; i += blockDim.x) {
      emit[i] = i < L ? 0.0f : x(i - L);
      hist[i] = x(i);
    }
    for (int i = threadIdx.x; i < L; i += blockDim.x) {
      fix[i] = 0.0f;
      prev_tail[i] = x(chunk - L + i);
    }
  }
}

__global__ void __launch_bounds__(POST_THREADS)
emit_chunk_kernel(const float* __restrict__ wav, int n_have, int chunk, int L, int has_prev, float target_rms,
                  float silence_thr, const float* __restrict__ fade_in, float* __restrict__ prev_tail,
                  float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double scratch[POST_THREADS / 32 + 1];
  emit_chunk_body(wav, n_have, chunk, L, has_prev, target_rms, silence_thr, fade_in, prev_tail, out, scratch);
}

// The same chain for the n sessions of one session-pool batch (mc_pool_push_codes_emit), one CTA per batch item j:
//   wav       [n, ld]                    decoded windows, n_have samples each
//   table     [n][2]                     table[2j] = pool slot of item j (the table pool_roll_kernel reads)
//   prev_tails[max_sessions, L]          per-slot crossfade tails, updated in place
//   out       [n, 2*chunk + L]           item j's block in emit_chunk_kernel's layout
// has_prev is shared by the whole batch (the engine groups first chunks apart from continuing ones).
__global__ void __launch_bounds__(POST_THREADS)
emit_chunk_pool_kernel(const float* __restrict__ wav, long long ld, int n_have, const int* __restrict__ table, int chunk,
                       int L, int has_prev, float target_rms, float silence_thr, const float* __restrict__ fade_in,
                       float* __restrict__ prev_tails, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double scratch[POST_THREADS / 32 + 1];
  const int j = blockIdx.x;
  const long long slot = table[2 * j];
  emit_chunk_body(wav + j * ld, n_have, chunk, L, has_prev, target_rms, silence_thr, fade_in, prev_tails + slot * L,
                  out + static_cast<long long>(j) * (2 * chunk + L), scratch);
}

// The agent render of a whole stream in ONE launch (offline decode, mc_render_chunks), one CTA per chunk.  Chunk i's
// part of the recording needs its own normalised window and the first L samples of chunk i+1's window (the crossfade
// replaces its tail), but no earlier output: the prev_tail emit_chunk_kernel carries is always the last L samples of
// the predecessor's own window.  Scales use the same fixed-order block_sum_f64 and the mixes the same separate
// roundings as emit_chunk_kernel, so the result equals running that kernel chunk by chunk, bit for bit.
//   windows [n_chunks, ld]: row 0 = the first chunk (no preroll), rows i >= 1 = L preroll ++ chunk; the last row holds
//                           last_len new samples, the rest of it reads as zeros (pad_or_trim)
//   out     [(n_chunks - 1) * chunk + last_len]: np.concatenate(audio_history_ch1), aligned with the codes
__device__ __forceinline__ float render_row_scale(const float* __restrict__ w, int n, int want, float target_rms,
                                                  float silence_thr, double* scratch) {
  float scale = 1.0f;
  if (target_rms > 0.0f) {
    double ss = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const double v = static_cast<double>(w[i]);
      ss += v * v;
    }
    ss = block_sum_f64(ss, scratch);
    const float rms = sqrtf(static_cast<float>(ss / static_cast<double>(want)));
    if (rms >= silence_thr) scale = target_rms / rms;
  }
  return scale;
}

__global__ void __launch_bounds__(POST_THREADS)
emit_chunks_kernel(const float* __restrict__ windows, long long ld, int n_chunks, int chunk, int L, int last_len,
                   float target_rms, float silence_thr, const float* __restrict__ fade_in, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double scratch[POST_THREADS / 32 + 1];
  const int c = blockIdx.x;
  const bool last = c == n_chunks - 1;
  const int off = c ? L : 0;                                   // preroll samples in front of the chunk
  const int len = last ? last_len : chunk;
  const int n0 = off + len;                                    // valid samples of this row
  const float* w0 = windows + static_cast<long long>(c) * ld;
  const float s0 = render_row_scale(w0, n0, c ? chunk + L : chunk, target_rms, silence_thr, scratch);
  const float* w1 = last ? w0 : w0 + ld;
  const float s1 = last ? 1.0f
                        : render_row_scale(w1, L + (c + 1 == n_chunks - 1 ? last_len : chunk), chunk + L, target_rms,
                                           silence_thr, scratch);
  float* o = out + static_cast<long long>(c) * chunk;
  for (int k = threadIdx.x; k < len; k += blockDim.x) {
    float e = __fmul_rn(w0[off + k], s0);
    const int j = k - (chunk - L);
    // separate roundings like numpy's tail1 * fade_out + head2 * fade_in (no FMA contraction)
    if (!last && j >= 0) e = __fadd_rn(__fmul_rn(e, fade_in[L - 1 - j]), __fmul_rn(__fmul_rn(w1[j], s1), fade_in[j]));
    o[k] = e;
  }
}

// ids int64 [rows, n] (token ids; code = id - vocab_start) -> out[rows] = mean_j || table[code_j] - ref ||_2
// and, when mean_out != nullptr, mean_out[rows, 16] = mean_j table[code_j] (the silence embedding).
// One CTA per row.
__global__ void __launch_bounds__(POST_THREADS)
embed_distance_kernel(const long long* __restrict__ ids, int n, long long vocab_start, const float* __restrict__ table,
                      int K, const float* __restrict__ ref /*[16] or nullptr*/, float* __restrict__ dist_out,
                      float* __restrict__ mean_out) {
  __shared__ double scratch[POST_THREADS / 32 + 1];
  const long long* row = ids + static_cast<long long>(blockIdx.x) * n;
  float r[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) r[c] = ref ? __ldg(ref + c) : 0.0f;
  double dsum = 0.0;
  double esum[16];
#pragma unroll
  for (int c = 0; c < 16; ++c) esum[c] = 0.0;
  for (int j = threadIdx.x; j < n; j += blockDim.x) {
    long long code = row[j] - vocab_start;
    code = code < 0 ? 0 : (code >= K ? K - 1 : code);
    const float4* src = reinterpret_cast<const float4*>(table + code * 16);
    float e[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 v = __ldg(src + q);
      e[4 * q] = v.x; e[4 * q + 1] = v.y; e[4 * q + 2] = v.z; e[4 * q + 3] = v.w;
    }
    float ss = 0.0f;
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const float dlt = e[c] - r[c];
      ss = fmaf(dlt, dlt, ss);
      esum[c] += static_cast<double>(e[c]);
    }
    dsum += static_cast<double>(sqrtf(ss));
  }
  if (dist_out) {
    const double t = block_sum_f64(dsum, scratch);
    if (threadIdx.x == 0) dist_out[blockIdx.x] = static_cast<float>(t / static_cast<double>(n));
  }
  if (mean_out) {
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      const double t = block_sum_f64(esum[c], scratch);
      if (threadIdx.x == 0) mean_out[blockIdx.x * 16 + c] = static_cast<float>(t / static_cast<double>(n));
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Session pool (SURVEY §8 f2: TTS-server style multi-session batching, tts_server.py:59,158): the rolling contexts of
// up to max_sessions sessions live in one [slot][channel][cap] ping-pong buffer.  ONE launch rolls the contexts of
// the n sessions of a batch (kept tail of the old context ++ the staged new chunk, audio_tokenizer.py:72-74 /
// :111-113) and gathers them into the dense [n*C, ld] batch the encoder / decoder reads.
//   table[2j] = slot of batch item j, table[2j+1] = which of the two context buffers currently holds it
// `table` and `staged` may be PINNED HOST memory read in place (single sessions: one kernel instead of three copy nodes).
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
pool_roll_kernel(const int* __restrict__ table, int C, int cap, int old_len, int keep_old, int n_new, T* __restrict__ ctx0,
                 T* __restrict__ ctx1, const T* __restrict__ staged /*[n*C, cap]*/, T* __restrict__ batch, int batch_ld) {
  const int jc = blockIdx.y;                                   // batch row = j*C + c
  const int j = jc / C, c = jc - j * C;
  const int slot = table[2 * j], par = table[2 * j + 1];
  const T* src = (par ? ctx1 : ctx0) + (static_cast<long long>(slot) * C + c) * cap;
  T* dst = (par ? ctx0 : ctx1) + (static_cast<long long>(slot) * C + c) * cap;
  const T* st = staged + static_cast<long long>(jc) * cap;
  T* bt = batch != nullptr ? batch + static_cast<long long>(jc) * batch_ld : nullptr;   // NULL: the consumer reads the context itself
  const int new_len = keep_old + n_new;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < new_len; i += gridDim.x * blockDim.x) {
    const T v = i < keep_old ? src[old_len - keep_old + i] : st[i - keep_old];
    dst[i] = v;
    if (bt != nullptr) bt[i] = v;
  }
}

// ---------------------------------------------------------------------------------------------
// Ragged session-pool batches (mc_pool_push_*_ragged): the items' contexts differ in length.  The encoder and decoder
// are causal for window_right == 0, so every item's window starts at row 0 of the batch and reads zeros (audio) or
// code 0 (codes) past its own end; its frames are then bit-identical to its lone pass (DESIGN.md §4 "Warm-up prefixes").
//   rtable[4j .. 4j+3] = {slot, context buffer, old_len, new_len} of batch item j
// ---------------------------------------------------------------------------------------------
// pool_roll_kernel per item, plus the zero fill: batch row j*C + c = the item's new_len values, then zeros up to `width`
// (T_max samples or F_max frames).
template <typename T>
__global__ void __launch_bounds__(256)
pool_roll_ragged_kernel(const int* __restrict__ rtable, int C, int cap, int n_new, T* __restrict__ ctx0, T* __restrict__ ctx1,
                        const T* __restrict__ staged /*[n*C, cap]*/, T* __restrict__ batch, int batch_ld, int width) {
  const int jc = blockIdx.y;
  const int j = jc / C, c = jc - j * C;
  const int slot = rtable[4 * j], par = rtable[4 * j + 1], old_len = rtable[4 * j + 2], new_len = rtable[4 * j + 3];
  const int keep_old = new_len - n_new;
  const T* src = (par ? ctx1 : ctx0) + (static_cast<long long>(slot) * C + c) * cap;
  T* dst = (par ? ctx0 : ctx1) + (static_cast<long long>(slot) * C + c) * cap;
  const T* st = staged + static_cast<long long>(jc) * cap;
  T* bt = batch + static_cast<long long>(jc) * batch_ld;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < width; i += gridDim.x * blockDim.x) {
    if (i < new_len) {
      const T v = i < keep_old ? src[old_len - keep_old + i] : st[i - keep_old];
      dst[i] = v;
      bt[i] = v;
    } else {
      bt[i] = T(0);
    }
  }
}

// Encode: z [n*C, rows, dq] holds the last `rows` frames of every F_max-frame window; item j keeps its own last `keep`
// frames, rows [F_j - keep, F_j) of its window with F_j = ceil(new_len_j / hop).  out [n*C, keep, dq], dense for the VQ.
__global__ void __launch_bounds__(256)
pool_gather_rows_ragged_kernel(const float* __restrict__ z, const int* __restrict__ rtable, int C, int rows, int F_max, int keep,
                               int dq, int hop, float* __restrict__ out) {
  const int jc = blockIdx.y, j = jc / C;
  const int F_j = (rtable[4 * j + 3] + hop - 1) / hop;
  const int r0 = rows - (F_max - F_j) - keep;
  const float* src = z + (static_cast<long long>(jc) * rows + r0) * dq;
  float* dst = out + static_cast<long long>(jc) * keep * dq;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < keep * dq; e += gridDim.x * blockDim.x) dst[e] = src[e];
}

// Decode: wav [n*C, ld] holds the last ld samples of every F_max*hop-sample window; item j keeps
// k_j = min(keep, new_len_j*hop) samples ending at its own end.  out [n*C, keep] (pinned host memory): the k_j samples at
// the row start, zeros after them.
__global__ void __launch_bounds__(256)
pool_gather_samples_ragged_kernel(const float* __restrict__ wav, long long ld, const int* __restrict__ rtable, int C, int total_max,
                                  int hop, int keep, float* __restrict__ out) {
  const int jc = blockIdx.y, j = jc / C;
  const int total_j = rtable[4 * j + 3] * hop;
  const int k = min(keep, total_j);
  const long long off = ld - (total_max - total_j) - k;
  const float* w = wav + jc * ld + off;
  float* o = out + static_cast<long long>(jc) * keep;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < keep; i += gridDim.x * blockDim.x) o[i] = i < k ? w[i] : 0.0f;
}

// emit_chunk_pool_kernel for a ragged batch: wav as for pool_gather_samples_ragged_kernel.  Item j's decoded samples are
// the last min(new_len_j*hop, chunk + L) of its window: chunk + L for a continuing chunk, chunk for a first one (the host
// checks that these agree with each slot's state), so has_prev and n_have are per item.
__global__ void __launch_bounds__(POST_THREADS)
emit_chunk_pool_ragged_kernel(const float* __restrict__ wav, long long ld, const int* __restrict__ rtable, int total_max, int hop,
                              int chunk, int L, float target_rms, float silence_thr, const float* __restrict__ fade_in,
                              float* __restrict__ prev_tails, float* __restrict__ out) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ double scratch[POST_THREADS / 32 + 1];
  const int j = blockIdx.x;
  const long long slot = rtable[4 * j];
  const int total_j = rtable[4 * j + 3] * hop;
  const int keep = min(total_j, chunk + L);
  const long long off = ld - (total_max - total_j) - keep;
  // keep == chunk + L <=> a continuing chunk: mc_pool_push_codes_emit_ragged rejects any slot whose keep disagrees with
  // its state (first chunk: keep == chunk), and mc_pool_set_emit enforces L >= 1, so the two cases never coincide
  emit_chunk_body(wav + j * ld + off, keep, chunk, L, keep == chunk + L ? 1 : 0, target_rms, silence_thr, fade_in,
                  prev_tails + slot * L, out + static_cast<long long>(j) * (2 * chunk + L), scratch);
}

}  // namespace mc
