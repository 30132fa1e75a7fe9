// Fused sliding-window attention on tcgen05, head_dim 64, causal window (keys j in [i-wl, i], wl <= 32).
//
//   TMA   Q[128x64], K[NKVx64], V[NKVx64] per (window, head, 128-query tile) through a ring of stages
//   UMMA  S = Q K^T            128 x NKV x 64 -> TMEM                    (K-major A and B)
//   SIMT  mask + softmax from TMEM, one thread per query row; P (bf16 pairs) goes back into TENSOR memory over the
//         dead S columns (v4, default) or into a 128B-swizzled shared-memory tile (v3, kept for A/B runs)
//   UMMA  O = P V              128 x 64 x NKV                             (A from TMEM in v4; B = V, MN-major)
//   SIMT  O / rowsum -> bf16 -> global
//
// S and P never touch HBM.  A window of <= 128 frames (every streaming / offline window: 100) is a single tile with
// NKV = 128; longer one-shot inputs tile along F with a 32-key halo (NKV = 160).  Round 1's first two versions (one
// item per CTA; two-slot pipeline without staged loads) were removed in round 2: v3 and v4 compute the same values in
// the same order (tests/test_gpu_ops.py keeps v4 == v3 bit for bit, and both against the SIMT cross-check kernel).
#pragma once
#include "engine_common.cuh"
#include "gemm_sm100.cuh"

namespace mc {

constexpr int ATT_BQ = 128;    // queries per CTA
constexpr int ATT_HALO = 32;   // keys before the first query
constexpr int ATT_SMEM_Q = ATT_BQ * 128;        // 16384
constexpr int ATT2_TMEM_COLS = 512;             // the persistent kernels allocate the whole tensor memory of their SM

inline bool attn_sm100_supported(int wl, int wr) { return wr == 0 && wl <= ATT_HALO; }

// Softmax details shared by v3 / v4: each softmax thread needs only the 64 score columns its row can see, read once
// from TMEM; masking is branch-free (masked scores become -inf, exp2 gives 0) and the row sum is accumulated strictly in
// ascending key order, so results do not depend on where a window was cut for dead-output elimination (adding the exact
// zeros of masked keys is a no-op); P*V sums keys in 16-key UMMA groups.
//
// ATTENTION CUTS.  The row sum adds keys in pairs and P*V in 16-key groups, both counted from the first column of the
// tile, so a frame must land at the same column mod 16 as in the full-window pass.  A window that dead-output
// elimination cut to its last F rows (F_full - F frames dropped) is therefore laid out with phase = (F_full - F) mod 16
// extra rows in front: Q and K/V tiles start `phase` rows before the window, i.e. at the previous window's last rows
// (finite values written by the same QKV GEMM) or, for the first window, in TMA's out-of-bounds zero fill.  Those
// columns are masked like any key before frame 0, and those query rows are never stored.  Every kept row then sees the
// same key groups, in the same order, with the same values as in the full pass: results are bit-identical at any cut.
//
// =============================================================================================

// v3: v2 with the operand loads decoupled from the compute slots.
//   * Q/K/V tiles travel through their own ring of TMA stages (3 deep for single-tile windows), so two
//     items are always in flight towards an SM while a third is being consumed — v2 could only request
//     an item's operands once the slot that would compute it had drained, which exposed the full
//     L2/HBM latency every second item (ncu: 34 % DRAM, 16 % tensor, nothing saturated).
//   * windows of <= 128 frames (every streaming and offline window: 100) are one query tile with
//     nothing before it, so NKV = 128 keys without the halo: 48 KB instead of 56 KB per item and S is
//     128 x 128.
//   * a thread's live P columns depend only on its row, so the P tiles are zeroed ONCE and each item
//     writes only its 64 live columns (128 B per row instead of 320 B).
//   * a compute slot needs only NKV TMEM columns: O = P*V is accumulated over the slot's own S columns (dead once
//     P is written).  The slot / stage counts are template constants (Att3Cfg); a 3-slot x 2-stage variant was
//     measured slower than 2 x 3 (see Att3Cfg).
//   warps 4g..4g+3  softmax + output of slot g     warp 4*slots  TMA producer     warp 4*slots+1  MMA issuer
//   kv_full[st] (tx) / kv_free[st] (commit after P*V)    s_full, p_full, o_full, slot_free per slot
// Arithmetic (mask, ex2, ascending-key row sum, bf16 P, 16-key UMMA groups) is v2's, so results are
// bit-identical to v2 and independent of where a window was cut for dead-output elimination.
//
// v4 (attention_window_sm100_v4_kernel, the default) is v3 with P kept in TENSOR memory: the softmax warps write
// their row of P (bf16 pairs) with tcgen05.st over the slot's dead S columns and P*V reads its A operand from
// there (tcgen05.mma with a TMEM A operand).  No P tile, no generic->async proxy fence and no A-operand re-read
// from shared memory per dispatch; the freed 64 KB go into a fourth TMA stage, and a slot is 128 TMEM columns,
// so three softmax groups fit.  Same values in the same order -> bit-identical to v3 / v2 (tested).
// =============================================================================================
template <int NKV>
struct Att3Cfg {
  static constexpr int kHalo = NKV - ATT_BQ;                        // 0 or 32 keys before the first query
  static constexpr int kStageBytes = ATT_SMEM_Q + 2 * NKV * 128;   // Q + K + V
  static constexpr int kPAtoms = (NKV + 63) / 64;
  static constexpr int kPBytes = kPAtoms * ATT_BQ * 128;
  // compute slots (one softmax group of 4 warps, one P tile and NKV TMEM columns each; O = P*V is accumulated over
  // the slot's own S columns, which are dead once P has been written) and TMA stages
  // measured at M = 102 400: 2 slots x 3 stages 1.46 ms per layer-launch set, 3 slots x 2 stages 1.81 ms — the
  // depth of the load ring matters more than a third softmax group, and both do not fit in 227 KB
  static constexpr int kSlots = 2;
  static constexpr int kStages = (NKV == 128) ? 3 : 2;
  static constexpr int kThreads = (4 * kSlots + 2) * 32;
  static constexpr int kSmemBytes = kStages * kStageBytes + kSlots * kPBytes + 256 + 1024;
  static_assert(kSlots * NKV <= 512, "TMEM columns");
  static_assert(kSmemBytes <= 232448, "shared memory");
};

template <int NKV>
__global__ void __launch_bounds__(Att3Cfg<NKV>::kThreads, 1)
attention_window_sm100_v3_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_kv,
                                 __nv_bfloat16* __restrict__ out, int B, int F, int H, int wl, int out_rows,
                                 int phase, float scale_log2e) {
  using Cfg = Att3Cfg<NKV>;
  constexpr int NST = Cfg::kStages;
  constexpr int NSL = Cfg::kSlots;
  constexpr int TMA_WARP = 4 * NSL, MMA_WARP = 4 * NSL + 1;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* p_base = smem + NST * Cfg::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(p_base + NSL * Cfg::kPBytes);
  uint64_t* kv_full = bars;             // [NST]
  uint64_t* kv_free = bars + NST;       // [NST]
  uint64_t* s_full = bars + 2 * NST;    // [NSL]
  uint64_t* p_full = s_full + NSL;      // [NSL]
  uint64_t* o_full = p_full + NSL;      // [NSL]
  uint64_t* slot_free = o_full + NSL;   // [NSL]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(slot_free + NSL);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = H * 64;
  const int Fp = F + phase;   // tile layout of a window: `phase` masked rows in front of its F rows (see ATTENTION CUTS)
  const int first_out = Fp - out_rows;
  const int q_tiles = (Fp + ATT_BQ - 1) / ATT_BQ;
  const int first_tile = first_out / ATT_BQ;
  const int kept_tiles = q_tiles - first_tile;
  const int n_items = B * H * kept_tiles;
  const int my_items = (n_items > static_cast<int>(blockIdx.x)) ? (n_items - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_kv);
    for (int s = 0; s < NST; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_free[s], 1);
    }
    for (int s = 0; s < NSL; ++s) {
      mbar_init(&s_full[s], 1);
      mbar_init(&p_full[s], 4);
      mbar_init(&o_full[s], 1);
      mbar_init(&slot_free[s], 4);
    }
    fence_mbar_init();
  }
  if (warp == MMA_WARP) {
    tmem_alloc(tmem_ptr, ATT2_TMEM_COLS);
    tmem_relinquish();
  }
  // P tiles start as zeros; only live columns are ever rewritten
  for (int i = threadIdx.x; i < NSL * Cfg::kPBytes / 16; i += Cfg::kThreads)
    reinterpret_cast<uint4*>(p_base)[i] = make_uint4(0, 0, 0, 0);
  fence_proxy_async_smem();
  pdl_launch_dependents();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_wait();

  if (warp == TMA_WARP) {
    if (lane == 0) {
      for (int it = 0; it < my_items; ++it) {
        const int item = blockIdx.x + it * gridDim.x;
        const int st = it % NST;
        const uint32_t use = (it / NST) & 1;
        const int qt = first_tile + item % kept_tiles;
        const int h = (item / kept_tiles) % H;
        const int b = item / (kept_tiles * H);
        uint8_t* stage = smem + st * Cfg::kStageBytes;
        mbar_wait(&kv_free[st], use ^ 1);
        mbar_arrive_expect_tx(&kv_full[st], Cfg::kStageBytes);
        const int row_q = b * F - phase + qt * ATT_BQ;
        tma_load_2d(stage, &map_q, &kv_full[st], h * 64, row_q);
        tma_load_2d(stage + ATT_SMEM_Q, &map_kv, &kv_full[st], d + h * 64, row_q - Cfg::kHalo);
        tma_load_2d(stage + ATT_SMEM_Q + NKV * 128, &map_kv, &kv_full[st], 2 * d + h * 64, row_q - Cfg::kHalo);
      }
    }
  } else if (warp == MMA_WARP) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(ATT_BQ, NKV, 0, 0);
      constexpr uint32_t idesc_o = umma_idesc_bf16(ATT_BQ, 64, 0, 1);
      // slot s serves items s, s+NSL, ...: S(it) -> P*V(it) -> S(it+NSL) ...; the single issuing thread polls all
      // slots and issues whatever is ready, so one slot's MMAs overlap the others' softmax.
      int cur[NSL];
      bool need_pv[NSL];
#pragma unroll
      for (int s = 0; s < NSL; ++s) { cur[s] = s; need_pv[s] = false; }
      int next_s = 0;
      int remaining = 2 * my_items;
      const long long t0 = clock64();
      while (remaining > 0) {
#pragma unroll
        for (int s = 0; s < NSL; ++s) {
          const int it = cur[s];
          if (it >= my_items) continue;
          const int st = it % NST;
          const uint32_t st_use = (it / NST) & 1;
          const uint32_t use = (it / NSL) & 1;
          uint8_t* stage = smem + st * Cfg::kStageBytes;
          if (!need_pv[s]) {
            // S steps are issued strictly in item order: a parity wait is only unambiguous one phase ahead, and with
            // fewer TMA stages than slots an out-of-order poll of kv_full[st] would see the PREVIOUS fill's phase
            if (it != next_s) continue;
            if (!mbar_try_wait(&slot_free[s], use ^ 1)) continue;   // previous item of this slot read its S and O
            if (!mbar_try_wait(&kv_full[st], st_use)) continue;
            tc_fence_after();
            const uint64_t qdesc = umma_smem_desc_sw128(smem_u32(stage), 1024, 16);
            const uint64_t kdesc = umma_smem_desc_sw128(smem_u32(stage + ATT_SMEM_Q), 1024, 16);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16_ss(tmem_base + s * NKV, qdesc + 2 * k, kdesc + 2 * k, idesc_s, k != 0);
            umma_commit(&s_full[s]);
            need_pv[s] = true;
            ++next_s;
            --remaining;
          } else {
            if (!mbar_try_wait(&p_full[s], use)) continue;
            tc_fence_after();
            uint8_t* sV = stage + ATT_SMEM_Q + NKV * 128;
            uint8_t* sP = p_base + s * Cfg::kPBytes;
#pragma unroll
            for (int k = 0; k < NKV / 16; ++k) {
              const uint64_t pdesc = umma_smem_desc_sw128(smem_u32(sP + (k >> 2) * (ATT_BQ * 128)) + (k & 3) * 32, 1024, 16);
              const uint64_t vdesc = umma_smem_desc_sw128(smem_u32(sV) + k * 2048, 1024, 1024);
              umma_bf16_ss(tmem_base + s * NKV, pdesc, vdesc, idesc_o, k != 0);   // O over the slot's (dead) S columns
            }
            umma_commit(&o_full[s]);
            umma_commit(&kv_free[st]);     // Q, K and V of this stage are consumed once these MMAs retire
            need_pv[s] = false;
            cur[s] += NSL;
            --remaining;
          }
        }
        if (clock64() - t0 > 8000000000LL) {
          printf("attention v3: MMA issuer timeout, block %d\n", blockIdx.x);
          __trap();
        }
      }
    }
  } else {
    const int s = warp >> 2;                   // softmax group = compute slot
    const int q = warp & 3;                    // TMEM lane quarter
    const int r = q * 32 + lane;               // query row inside the tile
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    uint8_t* sP = p_base + s * Cfg::kPBytes;
    const uint32_t tmem_s = tmem_base + s * NKV;
    const uint32_t tmem_o = tmem_s;            // P*V accumulates over S, which every warp has finished reading by then
    // rows of this warp see key columns [col_base, col_base + 64); without a halo the first 32 of warp 0 do not exist
    const int col_base = q * 32 + Cfg::kHalo - 32;
    for (int it = s; it < my_items; it += NSL) {
      const int item = blockIdx.x + it * gridDim.x;
      const uint32_t use = (it / NSL) & 1;
      const int qt = first_tile + item % kept_tiles;
      const int h = (item / kept_tiles) % H;
      const int b = item / (kept_tiles * H);
      const int q0 = qt * ATT_BQ;
      const int qi = q0 + r;

      mbar_wait(&s_full[s], use);
      tc_fence_after();
      uint32_t raw0[32], raw1[32];
      if (col_base >= 0) tmem_ld_32x32b_x32(tmem_s + lane_addr + col_base, raw0);
      tmem_ld_32x32b_x32(tmem_s + lane_addr + col_base + 32, raw1);
      tmem_ld_wait();
      const int c_lo = max(r + Cfg::kHalo - wl, Cfg::kHalo - q0 + phase) - col_base;   // relative to col_base
      const int c_hi = (qi < Fp) ? (r + Cfg::kHalo - col_base) : -1;
      float sc[64];
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        sc[j] = (col_base >= 0 && j >= c_lo && j <= c_hi) ? __uint_as_float(raw0[j]) * scale_log2e : -INFINITY;
        sc[32 + j] = (j + 32 >= c_lo && j + 32 <= c_hi) ? __uint_as_float(raw1[j]) * scale_log2e : -INFINITY;
      }
#pragma unroll
      for (int j = 0; j < 64; j += 2) mx = fmax3(mx, sc[j], sc[j + 1]);
      const float mref = (mx == -INFINITY) ? 0.0f : mx;
      float sum = 0.0f;
      uint32_t pk[32];
#pragma unroll
      for (int j = 0; j < 64; j += 2) {   // ascending keys, one accumulator
        float p0, p1;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p0) : "f"(sc[j] - mref));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p1) : "f"(sc[j + 1] - mref));
        sum += p0 + p1;
        pk[j >> 1] = pack_bf16x2(p0, p1);
      }
      // the two live 32-key chunks of this row (everything else in the P tile stays zero)
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int c0 = col_base + 32 * half;
        if (c0 < 0) continue;              // warp-uniform
        uint8_t* atom = sP + (c0 >> 6) * (ATT_BQ * 128) + r * 128;
        const int chunk0 = (c0 & 63) >> 3;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const uint4 w = make_uint4(pk[16 * half + 4 * u], pk[16 * half + 4 * u + 1], pk[16 * half + 4 * u + 2],
                                     pk[16 * half + 4 * u + 3]);
          *reinterpret_cast<uint4*>(atom + (((chunk0 + u) ^ (r & 7)) << 4)) = w;
        }
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[s]);

      mbar_wait(&o_full[s], use);
      tc_fence_after();
      tmem_ld_32x32b_x32(tmem_o + lane_addr, raw0);
      tmem_ld_32x32b_x32(tmem_o + lane_addr + 32, raw1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&slot_free[s]);   // S and O of this slot may be overwritten
      if (qi < Fp && qi >= first_out) {
        const float inv = 1.0f / sum;
        __nv_bfloat16* o = out + (static_cast<long long>(b) * out_rows + (qi - first_out)) * d + h * 64;
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint4 w;
          w.x = pack_bf16x2(__uint_as_float(raw0[j]) * inv, __uint_as_float(raw0[j + 1]) * inv);
          w.y = pack_bf16x2(__uint_as_float(raw0[j + 2]) * inv, __uint_as_float(raw0[j + 3]) * inv);
          w.z = pack_bf16x2(__uint_as_float(raw0[j + 4]) * inv, __uint_as_float(raw0[j + 5]) * inv);
          w.w = pack_bf16x2(__uint_as_float(raw0[j + 6]) * inv, __uint_as_float(raw0[j + 7]) * inv);
          *reinterpret_cast<uint4*>(o + j) = w;
        }
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint4 w;
          w.x = pack_bf16x2(__uint_as_float(raw1[j]) * inv, __uint_as_float(raw1[j + 1]) * inv);
          w.y = pack_bf16x2(__uint_as_float(raw1[j + 2]) * inv, __uint_as_float(raw1[j + 3]) * inv);
          w.z = pack_bf16x2(__uint_as_float(raw1[j + 4]) * inv, __uint_as_float(raw1[j + 5]) * inv);
          w.w = pack_bf16x2(__uint_as_float(raw1[j + 6]) * inv, __uint_as_float(raw1[j + 7]) * inv);
          *reinterpret_cast<uint4*>(o + 32 + j) = w;
        }
      }
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, ATT2_TMEM_COLS);
  }
}

template <int NKV>
struct Att4Cfg {
  static constexpr int kHalo = NKV - ATT_BQ;                        // 0 or 32 keys before the first query
  static constexpr int kStageBytes = ATT_SMEM_Q + 2 * NKV * 128;   // Q + K + V
  // P never touches shared memory: the softmax warps write it (bf16 pairs) into the slot's tensor-memory columns
  // [0, NKV/2) with tcgen05.st and P*V reads its A operand from there; O accumulates in columns [NKV/2, NKV/2 + 64).
  // Both alias the slot's S columns, which are dead by then.  The 64-96 KB of P tiles become a deeper load ring.
  static constexpr int kPCols = NKV / 2;
  // measured at M = 102 400 (NKV = 128, 4 stages): 2 slots 161 us, 3 slots 149 us, 4 slots 162 us (register cap 96);
  // the shared-memory-P kernel (v3, 2 slots x 3 stages) 165 us; HBM floor 128 us
  static constexpr int kSlots = 3;
  static constexpr int kStages = (NKV == 128) ? 4 : 3;
  static constexpr int kThreads = (4 * kSlots + 2) * 32;
  static constexpr int kSmemBytes = kStages * kStageBytes + 256 + 1024;
  static_assert(kSlots * NKV <= 512, "TMEM columns");
  static_assert(kSmemBytes <= 232448, "shared memory");
};

template <int NKV>
__global__ void __launch_bounds__(Att4Cfg<NKV>::kThreads, 1)
attention_window_sm100_v4_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_kv,
                                 __nv_bfloat16* __restrict__ out, int B, int F, int H, int wl, int out_rows,
                                 int phase, float scale_log2e) {
  using Cfg = Att4Cfg<NKV>;
  constexpr int NST = Cfg::kStages;
  constexpr int NSL = Cfg::kSlots;
  constexpr int TMA_WARP = 4 * NSL, MMA_WARP = 4 * NSL + 1;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NST * Cfg::kStageBytes);
  uint64_t* kv_full = bars;             // [NST]
  uint64_t* kv_free = bars + NST;       // [NST]
  uint64_t* s_full = bars + 2 * NST;    // [NSL]
  uint64_t* p_full = s_full + NSL;      // [NSL]
  uint64_t* o_full = p_full + NSL;      // [NSL]
  uint64_t* slot_free = o_full + NSL;   // [NSL]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(slot_free + NSL);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = H * 64;
  const int Fp = F + phase;   // tile layout of a window: `phase` masked rows in front of its F rows (see ATTENTION CUTS)
  const int first_out = Fp - out_rows;
  const int q_tiles = (Fp + ATT_BQ - 1) / ATT_BQ;
  const int first_tile = first_out / ATT_BQ;
  const int kept_tiles = q_tiles - first_tile;
  const int n_items = B * H * kept_tiles;
  const int my_items = (n_items > static_cast<int>(blockIdx.x)) ? (n_items - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_q);
    tma_prefetch_desc(&map_kv);
    for (int s = 0; s < NST; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_free[s], 1);
    }
    for (int s = 0; s < NSL; ++s) {
      mbar_init(&s_full[s], 1);
      mbar_init(&p_full[s], 4);
      mbar_init(&o_full[s], 1);
      mbar_init(&slot_free[s], 4);
    }
    fence_mbar_init();
  }
  if (warp == MMA_WARP) {
    tmem_alloc(tmem_ptr, ATT2_TMEM_COLS);
    tmem_relinquish();
  }
  pdl_launch_dependents();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_wait();

  if (warp == TMA_WARP) {
    if (lane == 0) {
      for (int it = 0; it < my_items; ++it) {
        const int item = blockIdx.x + it * gridDim.x;
        const int st = it % NST;
        const uint32_t use = (it / NST) & 1;
        const int qt = first_tile + item % kept_tiles;
        const int h = (item / kept_tiles) % H;
        const int b = item / (kept_tiles * H);
        uint8_t* stage = smem + st * Cfg::kStageBytes;
        mbar_wait(&kv_free[st], use ^ 1);
        mbar_arrive_expect_tx(&kv_full[st], Cfg::kStageBytes);
        const int row_q = b * F - phase + qt * ATT_BQ;
        tma_load_2d(stage, &map_q, &kv_full[st], h * 64, row_q);
        tma_load_2d(stage + ATT_SMEM_Q, &map_kv, &kv_full[st], d + h * 64, row_q - Cfg::kHalo);
        tma_load_2d(stage + ATT_SMEM_Q + NKV * 128, &map_kv, &kv_full[st], 2 * d + h * 64, row_q - Cfg::kHalo);
      }
    }
  } else if (warp == MMA_WARP) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(ATT_BQ, NKV, 0, 0);
      constexpr uint32_t idesc_o = umma_idesc_bf16(ATT_BQ, 64, 0, 1);
      // slot s serves items s, s+NSL, ...: S(it) -> P*V(it) -> S(it+NSL) ...; the single issuing thread polls all
      // slots and issues whatever is ready, so one slot's MMAs overlap the others' softmax.
      int cur[NSL];
      bool need_pv[NSL];
#pragma unroll
      for (int s = 0; s < NSL; ++s) { cur[s] = s; need_pv[s] = false; }
      int next_s = 0;
      int remaining = 2 * my_items;
      const long long t0 = clock64();
      while (remaining > 0) {
#pragma unroll
        for (int s = 0; s < NSL; ++s) {
          const int it = cur[s];
          if (it >= my_items) continue;
          const int st = it % NST;
          const uint32_t st_use = (it / NST) & 1;
          const uint32_t use = (it / NSL) & 1;
          uint8_t* stage = smem + st * Cfg::kStageBytes;
          if (!need_pv[s]) {
            // S steps are issued strictly in item order: a parity wait is only unambiguous one phase ahead, and with
            // fewer TMA stages than slots an out-of-order poll of kv_full[st] would see the PREVIOUS fill's phase
            if (it != next_s) continue;
            if (!mbar_try_wait(&slot_free[s], use ^ 1)) continue;   // previous item of this slot read its S and O
            if (!mbar_try_wait(&kv_full[st], st_use)) continue;
            tc_fence_after();
            const uint64_t qdesc = umma_smem_desc_sw128(smem_u32(stage), 1024, 16);
            const uint64_t kdesc = umma_smem_desc_sw128(smem_u32(stage + ATT_SMEM_Q), 1024, 16);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16_ss(tmem_base + s * NKV, qdesc + 2 * k, kdesc + 2 * k, idesc_s, k != 0);
            umma_commit(&s_full[s]);
            need_pv[s] = true;
            ++next_s;
            --remaining;
          } else {
            if (!mbar_try_wait(&p_full[s], use)) continue;
            tc_fence_after();
            uint8_t* sV = stage + ATT_SMEM_Q + NKV * 128;
#pragma unroll
            for (int k = 0; k < NKV / 16; ++k) {
              // A: 16 keys = 8 packed columns of the slot's P region; B: V rows are keys, 16 keys = 2048 bytes per step
              const uint64_t vdesc = umma_smem_desc_sw128(smem_u32(sV) + k * 2048, 1024, 1024);
              umma_bf16_ts(tmem_base + s * NKV + Cfg::kPCols, tmem_base + s * NKV + k * 8, vdesc, idesc_o, k != 0);
            }
            umma_commit(&o_full[s]);
            umma_commit(&kv_free[st]);     // Q, K and V of this stage are consumed once these MMAs retire
            need_pv[s] = false;
            cur[s] += NSL;
            --remaining;
          }
        }
        if (clock64() - t0 > 8000000000LL) {
          printf("attention v3: MMA issuer timeout, block %d\n", blockIdx.x);
          __trap();
        }
      }
    }
  } else {
    const int s = warp >> 2;                   // softmax group = compute slot
    const int q = warp & 3;                    // TMEM lane quarter
    const int r = q * 32 + lane;               // query row inside the tile
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t tmem_s = tmem_base + s * NKV;
    const uint32_t tmem_p = tmem_s;                      // P (bf16 pairs) over S columns [0, NKV/2)
    const uint32_t tmem_o = tmem_s + Cfg::kPCols;        // O over S columns [NKV/2, NKV/2 + 64)
    // rows of this warp see key columns [col_base, col_base + 64); without a halo the first 32 of warp 0 do not exist
    const int col_base = q * 32 + Cfg::kHalo - 32;
    for (int it = s; it < my_items; it += NSL) {
      const int item = blockIdx.x + it * gridDim.x;
      const uint32_t use = (it / NSL) & 1;
      const int qt = first_tile + item % kept_tiles;
      const int h = (item / kept_tiles) % H;
      const int b = item / (kept_tiles * H);
      const int q0 = qt * ATT_BQ;
      const int qi = q0 + r;

      mbar_wait(&s_full[s], use);
      tc_fence_after();
      uint32_t raw0[32], raw1[32];
      if (col_base >= 0) tmem_ld_32x32b_x32(tmem_s + lane_addr + col_base, raw0);
      tmem_ld_32x32b_x32(tmem_s + lane_addr + col_base + 32, raw1);
      tmem_ld_wait();
      const int c_lo = max(r + Cfg::kHalo - wl, Cfg::kHalo - q0 + phase) - col_base;   // relative to col_base
      const int c_hi = (qi < Fp) ? (r + Cfg::kHalo - col_base) : -1;
      float sc[64];
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        sc[j] = (col_base >= 0 && j >= c_lo && j <= c_hi) ? __uint_as_float(raw0[j]) * scale_log2e : -INFINITY;
        sc[32 + j] = (j + 32 >= c_lo && j + 32 <= c_hi) ? __uint_as_float(raw1[j]) * scale_log2e : -INFINITY;
      }
#pragma unroll
      for (int j = 0; j < 64; j += 2) mx = fmax3(mx, sc[j], sc[j + 1]);
      const float mref = (mx == -INFINITY) ? 0.0f : mx;
      float sum = 0.0f;
      uint32_t pk[32];
#pragma unroll
      for (int j = 0; j < 64; j += 2) {   // ascending keys, one accumulator
        float p0, p1;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p0) : "f"(sc[j] - mref));
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(p1) : "f"(sc[j + 1] - mref));
        sum += p0 + p1;
        pk[j >> 1] = pack_bf16x2(p0, p1);
      }
      // this row's P: NKV/2 packed columns in 16-column blocks; blocks (col_base/32) and (col_base/32 + 1) are live,
      // the others are zeros (S occupied these columns a moment ago, so they are rewritten for every item)
      {
        const uint32_t zeros[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        const int live0 = col_base / 32;                 // may be -1 (warp 0 without a halo)
#pragma unroll
        for (int blk = 0; blk < Cfg::kPCols / 16; ++blk) {
          const uint32_t taddr = tmem_p + lane_addr + blk * 16;
          if (blk == live0) {
            uint32_t w[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) w[u] = pk[u];
            tmem_st_32x32b_x16(taddr, w);
          } else if (blk == live0 + 1) {
            uint32_t w[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) w[u] = pk[16 + u];
            tmem_st_32x32b_x16(taddr, w);
          } else {
            tmem_st_32x32b_x16(taddr, zeros);
          }
        }
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[s]);

      mbar_wait(&o_full[s], use);
      tc_fence_after();
      tmem_ld_32x32b_x32(tmem_o + lane_addr, raw0);
      tmem_ld_32x32b_x32(tmem_o + lane_addr + 32, raw1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&slot_free[s]);   // S and O of this slot may be overwritten
      if (qi < Fp && qi >= first_out) {
        const float inv = 1.0f / sum;
        __nv_bfloat16* o = out + (static_cast<long long>(b) * out_rows + (qi - first_out)) * d + h * 64;
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint4 w;
          w.x = pack_bf16x2(__uint_as_float(raw0[j]) * inv, __uint_as_float(raw0[j + 1]) * inv);
          w.y = pack_bf16x2(__uint_as_float(raw0[j + 2]) * inv, __uint_as_float(raw0[j + 3]) * inv);
          w.z = pack_bf16x2(__uint_as_float(raw0[j + 4]) * inv, __uint_as_float(raw0[j + 5]) * inv);
          w.w = pack_bf16x2(__uint_as_float(raw0[j + 6]) * inv, __uint_as_float(raw0[j + 7]) * inv);
          *reinterpret_cast<uint4*>(o + j) = w;
        }
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint4 w;
          w.x = pack_bf16x2(__uint_as_float(raw1[j]) * inv, __uint_as_float(raw1[j + 1]) * inv);
          w.y = pack_bf16x2(__uint_as_float(raw1[j + 2]) * inv, __uint_as_float(raw1[j + 3]) * inv);
          w.z = pack_bf16x2(__uint_as_float(raw1[j + 4]) * inv, __uint_as_float(raw1[j + 5]) * inv);
          w.w = pack_bf16x2(__uint_as_float(raw1[j + 6]) * inv, __uint_as_float(raw1[j + 7]) * inv);
          *reinterpret_cast<uint4*>(o + 32 + j) = w;
        }
      }
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) {
    tc_fence_after();
    tmem_dealloc(tmem_base, ATT2_TMEM_COLS);
  }
}

template <int NKV>
inline int launch_attention_sm100_v4_nkv(mc_handle* h, const bf16* qkv, bf16* out, int B, int F, int out_rows,
                                         int phase, cudaStream_t stream) {
  using Cfg = Att4Cfg<NKV>;
  const mc_spec& s = h->spec;
  const int d = s.d_model;
  const CUtensorMap *mq, *mkv;
  MC_TRY(mc_internal::get_map_2d_bf16(h, qkv, (uint64_t)3 * d, (uint64_t)B * F, 64, ATT_BQ, &mq));
  MC_TRY(mc_internal::get_map_2d_bf16(h, qkv, (uint64_t)3 * d, (uint64_t)B * F, 64, NKV, &mkv));
  MC_TRY(mc_allow_smem(h, attention_window_sm100_v4_kernel<NKV>, Cfg::kSmemBytes));
  const int q_tiles = (F + phase + ATT_BQ - 1) / ATT_BQ;
  const long long items = (long long)B * s.n_heads * (q_tiles - (F + phase - out_rows) / ATT_BQ);
  if (items > INT_MAX) return h->fail(MC_ERR_ARG, "attention: too many tiles");
  const int grid = (int)std::min<long long>(items, h->num_sms);
  mc_launch(h, attention_window_sm100_v4_kernel<NKV>, dim3(grid), dim3(Cfg::kThreads), Cfg::kSmemBytes, stream, *mq, *mkv, out, B, F,
            s.n_heads, s.window_left, out_rows, phase, 0.125f * 1.4426950408889634f);
  MC_LAUNCH_CHECK(h, "attention_window_sm100_v4_kernel");
  return MC_OK;
}

template <int NKV>
inline int launch_attention_sm100_v3_nkv(mc_handle* h, const bf16* qkv, bf16* out, int B, int F, int out_rows,
                                         int phase, cudaStream_t stream) {
  using Cfg = Att3Cfg<NKV>;
  const mc_spec& s = h->spec;
  const int d = s.d_model;
  const CUtensorMap *mq, *mkv;
  MC_TRY(mc_internal::get_map_2d_bf16(h, qkv, (uint64_t)3 * d, (uint64_t)B * F, 64, ATT_BQ, &mq));
  MC_TRY(mc_internal::get_map_2d_bf16(h, qkv, (uint64_t)3 * d, (uint64_t)B * F, 64, NKV, &mkv));
  MC_TRY(mc_allow_smem(h, attention_window_sm100_v3_kernel<NKV>, Cfg::kSmemBytes));
  const int q_tiles = (F + phase + ATT_BQ - 1) / ATT_BQ;
  const long long items = (long long)B * s.n_heads * (q_tiles - (F + phase - out_rows) / ATT_BQ);
  if (items > INT_MAX) return h->fail(MC_ERR_ARG, "attention: too many tiles");
  const int grid = (int)std::min<long long>(items, h->num_sms);
  mc_launch(h, attention_window_sm100_v3_kernel<NKV>, dim3(grid), dim3(Cfg::kThreads), Cfg::kSmemBytes, stream, *mq, *mkv, out, B, F,
            s.n_heads, s.window_left, out_rows, phase, 0.125f * 1.4426950408889634f);
  MC_LAUNCH_CHECK(h, "attention_window_sm100_v3_kernel");
  return MC_OK;
}

// phase: rows in front of the window that complete its first 16-key group (0 .. 15; see ATTENTION CUTS)
inline int launch_attention_sm100_v3(mc_handle* h, const bf16* qkv, bf16* out, int B, int F, int out_rows, int phase,
                                     cudaStream_t stream) {
  if (phase < 0 || phase > 15) return h->fail(MC_ERR_ARG, "attention: cut phase %d is not in 0 .. 15", phase);
  const bool one_tile = F + phase <= ATT_BQ;
  if (h->attn_p_tmem) {
    if (one_tile) return launch_attention_sm100_v4_nkv<128>(h, qkv, out, B, F, out_rows, phase, stream);
    return launch_attention_sm100_v4_nkv<160>(h, qkv, out, B, F, out_rows, phase, stream);
  }
  if (one_tile) return launch_attention_sm100_v3_nkv<128>(h, qkv, out, B, F, out_rows, phase, stream);
  return launch_attention_sm100_v3_nkv<160>(h, qkv, out, B, F, out_rows, phase, stream);
}

}  // namespace mc
