// Corpus ingest on the device (SURVEY §8 a13 / f1: what _prep_audio_for_tokenization and the offline CLI do on the
// host in the reference — int16 -> float, librosa.to_mono, librosa.resample; audio_tokenizer.py:203-215).
//
// At ~5 400x real time per GPU the encoder consumes 350 MB/s of fp32 audio; the telephone corpora the reference
// encodes (CallHome / CallFriend / Fisher, encode_audio_gpu_1.sh:8) are 8 kHz mu-law or 16-bit stereo and must be
// resampled to 16 kHz first.  A host polyphase resampler delivers ~10 audio-minutes per core-second; here the raw
// container payload (1-2 bytes per sample) crosses PCIe and two HBM-bound kernels do the rest:
//
//   pcm_to_f32_kernel      interleaved PCM (u8 / s16 / s24 / s32 / f32 / f64 / mu-law / A-law) -> planar fp32 [C, n],
//                          optional mono mix (mean over channels, fp32, like np.mean(axis=0))
//   resample_poly_kernel   rational polyphase FIR: out[i] = sum_j h[(t % up) + j*up] * x[t / up - j], t = (i + pre)*down
//                          — scipy.signal.resample_poly's upfirdn with the same (pre-padded, up-scaled) taps, fp32
//                          accumulation in a fixed order (bit-reproducible)
//   f32_to_pcm_kernel      the way back for the offline decode: planar fp32 -> interleaved s16 / f32 PCM
#pragma once
#include "engine_common.cuh"

namespace mc {

enum : int { PCM_U8 = 0, PCM_S16 = 1, PCM_S24 = 2, PCM_S32 = 3, PCM_F32 = 4, PCM_F64 = 5, PCM_ULAW = 6, PCM_ALAW = 7 };

// G.711 expansions to 16-bit linear (the same tables libsndfile / sph2pipe produce)
__device__ __forceinline__ int ulaw_to_s16(unsigned char u) {
  u = ~u;
  const int t = (((u & 0x0F) << 3) + 0x84) << ((u & 0x70) >> 4);
  return (u & 0x80) ? (0x84 - t) : (t - 0x84);
}
__device__ __forceinline__ int alaw_to_s16(unsigned char a) {
  a ^= 0x55;
  int t = (a & 0x0F) << 4;
  const int seg = (a & 0x70) >> 4;
  if (seg == 0) t += 8;
  else if (seg == 1) t += 0x108;
  else t = (t + 0x108) << (seg - 1);
  return (a & 0x80) ? t : -t;
}

__device__ __forceinline__ float pcm_sample(const unsigned char* src, int fmt, long long idx, int big_endian) {
  switch (fmt) {
    case PCM_U8: return (static_cast<float>(src[idx]) - 128.0f) * (1.0f / 128.0f);
    case PCM_S16: {
      const unsigned char* p = src + idx * 2;
      const int v = big_endian ? static_cast<short>((p[0] << 8) | p[1]) : static_cast<short>((p[1] << 8) | p[0]);
      return static_cast<float>(v) * (1.0f / 32768.0f);
    }
    case PCM_S24: {
      const unsigned char* p = src + idx * 3;
      int v = big_endian ? ((p[0] << 16) | (p[1] << 8) | p[2]) : ((p[2] << 16) | (p[1] << 8) | p[0]);
      v = (v << 8) >> 8;
      return static_cast<float>(v) * (1.0f / 8388608.0f);
    }
    case PCM_S32: {
      const unsigned char* p = src + idx * 4;
      const int v = big_endian ? static_cast<int>((static_cast<unsigned>(p[0]) << 24) | (p[1] << 16) | (p[2] << 8) | p[3])
                               : static_cast<int>((static_cast<unsigned>(p[3]) << 24) | (p[2] << 16) | (p[1] << 8) | p[0]);
      return static_cast<float>(v) * (1.0f / 2147483648.0f);
    }
    case PCM_F32: {
      if (!big_endian) return reinterpret_cast<const float*>(src)[idx];
      return __uint_as_float(__byte_perm(reinterpret_cast<const unsigned*>(src)[idx], 0, 0x0123));
    }
    case PCM_F64: {
      if (!big_endian) return static_cast<float>(reinterpret_cast<const double*>(src)[idx]);
      const unsigned long long v = reinterpret_cast<const unsigned long long*>(src)[idx];
      const unsigned lo = __byte_perm(static_cast<unsigned>(v >> 32), 0, 0x0123), hi = __byte_perm(static_cast<unsigned>(v), 0, 0x0123);
      return static_cast<float>(__longlong_as_double(static_cast<long long>((static_cast<unsigned long long>(hi) << 32) | lo)));
    }
    case PCM_ULAW: return static_cast<float>(ulaw_to_s16(src[idx])) * (1.0f / 32768.0f);
    default: return static_cast<float>(alaw_to_s16(src[idx])) * (1.0f / 32768.0f);
  }
}

// src: interleaved frames [n][C] (sample (t, c) at index t*C + c).  out: planar [C_out, out_ld]; mix_mono: C_out = 1.
__global__ void __launch_bounds__(256)
pcm_to_f32_kernel(const unsigned char* __restrict__ src, int fmt, int big_endian, int C, long long n, int mix_mono,
                  float* __restrict__ out, long long out_ld) {
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < n; t += stride) {
    if (mix_mono) {
      float acc = 0.0f;
      for (int c = 0; c < C; ++c) acc += pcm_sample(src, fmt, t * C + c, big_endian);
      out[t] = acc / static_cast<float>(C);
    } else {
      for (int c = 0; c < C; ++c) out[c * out_ld + t] = pcm_sample(src, fmt, t * C + c, big_endian);
    }
  }
}

// The mirror of pcm_to_f32_kernel for the offline decode's writer: planar fp32 [C, in_ld] -> interleaved [frames][C] as
// PCM_S16 (clamp(rint(x * 32768), -32768, 32767), NaN -> 0: the exact inverse of the reference's / 32768 on int16
// input) or PCM_F32.  `out` may be PINNED HOST memory: the stores are the device-to-host copy, at half the bytes of fp32
// for 16-bit output, interleaved in the same pass.
__global__ void __launch_bounds__(256)
f32_to_pcm_kernel(const float* __restrict__ in, long long in_ld, int C, long long frames, int fmt, void* __restrict__ out) {
  const long long total = frames * C;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total; e += stride) {
    const long long t = e / C;
    const int c = static_cast<int>(e - t * C);
    const float x = in[c * in_ld + t];
    if (fmt == PCM_S16) {
      const float v = rintf(x * 32768.0f);
      reinterpret_cast<short*>(out)[e] = v != v ? 0 : static_cast<short>(fminf(fmaxf(v, -32768.0f), 32767.0f));
    } else {
      reinterpret_cast<float*>(out)[e] = x;
    }
  }
}

// x: planar [C, in_ld] with n_in valid samples per channel; h: [n_taps] (already scaled by `up` and left-padded by
// the alignment zeros); out: planar [C, out_ld], n_out samples per channel.
__global__ void __launch_bounds__(256)
resample_poly_kernel(const float* __restrict__ x, long long in_ld, int C, long long n_in, int up, int down,
                     const float* __restrict__ h, int n_taps, long long pre_remove, float* __restrict__ out,
                     long long out_ld, long long n_out) {
  const long long total = static_cast<long long>(C) * n_out;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total; e += stride) {
    const int c = static_cast<int>(e / n_out);
    const long long i = e - static_cast<long long>(c) * n_out;
    const long long t = (i + pre_remove) * down;
    const int phase = static_cast<int>(t % up);
    const long long base = t / up;
    const float* xc = x + c * in_ld;
    // taps k = phase + j*up < n_taps;  samples base - j in [0, n_in)
    long long j0 = base >= n_in ? base - (n_in - 1) : 0;
    long long j1 = (n_taps - 1 - phase) / up;            // last j with a tap
    if (base < j1) j1 = base;
    float acc = 0.0f;
    for (long long j = j0; j <= j1; ++j) acc = fmaf(__ldg(h + phase + j * up), __ldg(xc + (base - j)), acc);
    out[c * out_ld + i] = acc;
  }
}

// ---------------------------------------------------------------------------------------------
// Live-stream ingest of a session-pool push (mc_pool_push_pcm): every item of the batch is one client's raw chunk (s16 or
// f32, planar [channels][n_in], at its own rate) and becomes the item's fp32 rows of the pool's chunk staging at the
// codec's rate, which pool_roll_kernel / pool_roll_ragged_kernel then read as for mc_pool_push_audio.  Per item and
// output channel the values are bit for bit those of pcm_to_f32_kernel (mixing to mono when a mono pool gets several
// channels) followed by resample_poly_kernel on the same bytes: the same conversion and mean, and the same FMA order.
// ---------------------------------------------------------------------------------------------
constexpr int INGEST_TILE = 256;    // outputs per CTA
constexpr int INGEST_SPAN = 8192;   // input samples a CTA holds in shared memory (the host checks each plan's span fits)

struct PoolIngestItem {             // one per batch item, read in place from pinned host memory
  const float* taps;                // device taps of the item's rate (resample_poly_kernel's h); NULL: the codec's rate
  long long offset;                 // byte offset of the item's rows [channels][n_in] in the staged payload
  long long pre_remove;
  int format, channels, n_in, up, down, n_taps;
};

// Input samples a tile of INGEST_TILE outputs can read: (TILE - 1) * down / up + 1 bases, (n_taps - 1) / up older ones.
__host__ __device__ inline long long ingest_span(int up, int down, int n_taps) {
  return static_cast<long long>(INGEST_TILE - 1) * down / up + (n_taps - 1) / up + 2;
}

// grid (ceil(n_out / INGEST_TILE), n * C_out); out: [n * C_out][out_ld], row j * C_out + c.
__global__ void __launch_bounds__(256)
pool_ingest_kernel(const PoolIngestItem* __restrict__ items, const unsigned char* __restrict__ payload, int C_out, int n_out,
                   float* __restrict__ out, int out_ld) {
  __shared__ float xs[INGEST_SPAN];
  const int jc = blockIdx.y, j = jc / C_out, c = jc - j * C_out;
  const PoolIngestItem it = items[j];
  const unsigned char* src = payload + it.offset;
  const bool mix = C_out == 1 && it.channels > 1;            // a mono pool fed several channels: np.mean(axis=0) in fp32
  const long long row = mix ? 0 : static_cast<long long>(c) * it.n_in;
  auto sample = [&](long long t) -> float {
    if (!mix) return pcm_sample(src, it.format, row + t, 0);
    float acc = 0.0f;
    for (int k = 0; k < it.channels; ++k) acc += pcm_sample(src, it.format, static_cast<long long>(k) * it.n_in + t, 0);
    return acc / static_cast<float>(it.channels);
  };
  const long long i0 = static_cast<long long>(blockIdx.x) * INGEST_TILE;
  const long long i1 = min(i0 + INGEST_TILE, static_cast<long long>(n_out));
  float* o = out + static_cast<long long>(jc) * out_ld;
  if (it.taps == nullptr) {                                    // the codec's rate: conversion only
    for (long long i = i0 + threadIdx.x; i < i1; i += blockDim.x) o[i] = sample(i);
    return;
  }
  const int up = it.up, down = it.down, n_taps = it.n_taps;
  const long long n_in = it.n_in;
  // the tile reads input samples [lo, hi]: base - j with base = (i + pre) * down / up and 0 <= j <= (n_taps - 1) / up
  const long long lo = max(0LL, (i0 + it.pre_remove) * down / up - (n_taps - 1) / up);
  const long long hi = min(n_in - 1, (i1 - 1 + it.pre_remove) * down / up);
  for (long long t = lo + threadIdx.x; t <= hi; t += blockDim.x) xs[t - lo] = sample(t);
  __syncthreads();
  const float* __restrict__ h = it.taps;
  for (long long i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
    // resample_poly_kernel's loop, reading the converted samples from shared memory
    const long long t = (i + it.pre_remove) * down;
    const int phase = static_cast<int>(t % up);
    const long long base = t / up;
    long long j0 = base >= n_in ? base - (n_in - 1) : 0;
    long long j1 = (n_taps - 1 - phase) / up;
    if (base < j1) j1 = base;
    float acc = 0.0f;
#pragma unroll 8   // the tap loads of 8 steps in flight; the FMAs stay in resample_poly_kernel's order
    for (long long jj = j0; jj <= j1; ++jj) acc = fmaf(__ldg(h + phase + jj * up), xs[base - jj - lo], acc);
    o[i] = acc;
  }
}

}  // namespace mc
