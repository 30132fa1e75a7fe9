// Engine: sequences the kernels of one encode / decode pass over workspaces it owns and exports
// the C ABI of include/magicodec_b200.h.
#include "engine_common.cuh"

#include "attn_sm100.cuh"
#include "attn_vq_simt.cuh"
#include "elementwise.cuh"
#include "gemm_sm100.cuh"
#include "gemm_splitk_sm100.cuh"
#include "ingest.cuh"
#include "post_sm100.cuh"
#include "vq_sm100.cuh"

using namespace mc;
using namespace mc_internal;

namespace {

// ------------------------------------------------------------------- GEMM
struct GemmCall {
  const bf16* A; int64_t a_rows; int a_k_wrap;
  const bf16* W; const float* bias;
  int M, N, K, act, out_mode;
  void* out; int64_t ldo;
  int grp_in = INT_MAX, grp_valid = INT_MAX; int64_t grp_stride = 0, grp_off = 0;
  int rope_cols = 0, rope_period = 0, rope_offset = 0;
  int block_n = 0;  // 0 = choose
  const void* prefetch_ptr = nullptr;   // next GEMM's weights (split-K kernel: L2 prefetch)
  long long prefetch_bytes = 0;
  // fused RMSNorm (few-rows path, GemmParams): consumer / producer
  const float* row_stats = nullptr; int row_stats_n = 0;
  bf16* xb_out = nullptr; const float* xb_gamma = nullptr; float* stat_out = nullptr;
};

void fill_norm_fields(const mc_handle* h, const GemmCall& c, GemmParams& p) {
  p.row_stats = c.row_stats; p.row_stats_n = c.row_stats_n;
  p.norm_eps = h->spec.norm_eps; p.inv_norm_dim = c.K > 0 ? 1.0f / (float)c.K : 0.f;   // the consumer's K is the normalised width
  p.xb_out = c.xb_out; p.xb_gamma = c.xb_gamma; p.stat_out = c.stat_out;
}

template <int BN, int BM = GEMM_BM, int KPS = 1>
int launch_gemm_bn(mc_handle* h, const GemmCall& c, cudaStream_t stream) {
  const CUtensorMap *ma, *mb;
  MC_TRY(get_map_2d_bf16(h, c.A, (uint64_t)c.a_k_wrap, (uint64_t)c.a_rows, GEMM_BK, BM, &ma));
  MC_TRY(get_map_2d_bf16(h, c.W, (uint64_t)c.K, (uint64_t)c.N, GEMM_BK, BN, &mb));
  // plain (ungrouped) outputs leave through TMA: bf16 boxes of 64 columns, fp32 boxes of 32
  // 64-row tiles (16 rows per epilogue warp) and fused-norm producers use per-thread stores
  const bool tma_out = (c.grp_in == INT_MAX) && BM == GEMM_BM && c.xb_out == nullptr;
  const CUtensorMap* mo = ma;
  if (tma_out) {
    const int esize = c.out_mode == OUT_BF16 ? 2 : 4;
    MC_TRY(get_map_2d(h, c.out, esize, (uint64_t)c.N, (uint64_t)c.M, (uint64_t)c.ldo * esize, esize == 2 ? 64 : 32, 32, &mo));
  }
  GemmParams p;
  p.tma_store = tma_out ? 1 : 0;
  p.M = c.M; p.N = c.N; p.K = c.K; p.a_k_wrap = c.a_k_wrap;
  p.bias = c.bias; p.act = c.act; p.out_mode = c.out_mode; p.out = c.out; p.ldo = c.ldo;
  p.grp_in = c.grp_in; p.grp_valid = c.grp_valid; p.grp_stride = c.grp_stride; p.grp_off = c.grp_off;
  p.rope_cols = c.rope_cols; p.rope_period = c.rope_period; p.rope_offset = c.rope_offset;
  p.rope_ld = h->spec.max_positions;
  p.rope_cos = c.rope_period > 0 ? h->ptr<float>("rope.cos") : nullptr;
  p.rope_sin = c.rope_period > 0 ? h->ptr<float>("rope.sin") : nullptr;
  fill_norm_fields(h, c, p);
  MC_TRY(mc_allow_smem(h, (gemm_bf16_sm100_kernel<BN, BM, KPS>), GemmCfg<BN>::kSmemBytes));
  const int m_tiles = (c.M + BM - 1) / BM, n_tiles = (c.N + BN - 1) / BN;
  const int grid = std::min(m_tiles * n_tiles, h->num_sms);
  const double valid_rows = c.grp_in == INT_MAX ? (double)c.M : (double)c.M / c.grp_in * c.grp_valid;
  const double out_bytes = valid_rows * c.N * (c.out_mode == OUT_BF16 ? 2.0 : (c.out_mode == OUT_F32 ? 4.0 : 8.0));
  McProfScope prof(h, 0, 2.0 * valid_rows * c.N * c.K, valid_rows * c.a_k_wrap * 2.0 + (double)c.N * c.K * 2.0 + out_bytes, stream);
  mc_launch(h, gemm_bf16_sm100_kernel<BN, BM, KPS>, dim3(grid), dim3(GEMM_THREADS), GemmCfg<BN>::kSmemBytes, stream, *ma, *mb, *mo, p);
  MC_LAUNCH_CHECK(h, "gemm_bf16_sm100_kernel");
  return MC_OK;
}

// CTA-pair kernel: 256 x 256 tiles on 74 clusters of two CTAs
template <int EPI>
int launch_gemm_pair_epi(mc_handle* h, const GemmParams& p, const CUtensorMap* ma, const CUtensorMap* mb,
                         const CUtensorMap* mo, const CUtensorMap* mo2, int pairs, cudaStream_t stream) {
  constexpr int BN = 256;
  MC_TRY(mc_allow_smem(h, gemm2_bf16_sm100_kernel<BN, EPI>, Gemm2Cfg<BN, EPI>::kSmemBytes));
  mc_launch(h, gemm2_bf16_sm100_kernel<BN, EPI>, dim3(2 * pairs), dim3(GEMM_THREADS), Gemm2Cfg<BN, EPI>::kSmemBytes, stream, *ma, *mb,
            *mo, *mo2, p);
  MC_LAUNCH_CHECK(h, "gemm2_bf16_sm100_kernel");
  return MC_OK;
}

int launch_gemm_pair(mc_handle* h, const GemmCall& c, cudaStream_t stream) {
  constexpr int BN = 256;
  const CUtensorMap *ma, *mb;
  MC_TRY(get_map_2d_bf16(h, c.A, (uint64_t)c.a_k_wrap, (uint64_t)c.a_rows, GEMM_BK, GEMM_BM, &ma));
  MC_TRY(get_map_2d_bf16(h, c.W, (uint64_t)c.K, (uint64_t)c.N, GEMM_BK, BN / 2, &mb));
  // fused-RMSNorm producer: the specialised epilogue (x_old in through TMA) when its conditions hold, else per-thread stores
  const bool norm_fast = c.xb_out != nullptr && h->fast_epilogue && c.grp_in == INT_MAX && c.bias != nullptr && c.N % BN == 0 &&
                         c.out_mode == OUT_F32_RESIDUAL && c.act == ACT_NONE && c.rope_period == 0 && c.ldo == c.N;
  const bool tma_out = (c.grp_in == INT_MAX) && (c.xb_out == nullptr || norm_fast);
  const CUtensorMap* mo = ma;
  const CUtensorMap* mo2 = ma;
  if (tma_out) {
    const int esize = c.out_mode == OUT_BF16 ? 2 : 4;
    MC_TRY(get_map_2d(h, c.out, esize, (uint64_t)c.N, (uint64_t)c.M, (uint64_t)c.ldo * esize, esize == 2 ? 64 : 32, 32, &mo));
  }
  if (norm_fast) MC_TRY(get_map_2d(h, c.xb_out, 2, (uint64_t)c.N, (uint64_t)c.M, (uint64_t)c.N * 2, 64, 32, &mo2));
  GemmParams p;
  p.tma_store = tma_out ? 1 : 0;
  p.M = c.M; p.N = c.N; p.K = c.K; p.a_k_wrap = c.a_k_wrap;
  p.bias = c.bias; p.act = c.act; p.out_mode = c.out_mode; p.out = c.out; p.ldo = c.ldo;
  p.grp_in = c.grp_in; p.grp_valid = c.grp_valid; p.grp_stride = c.grp_stride; p.grp_off = c.grp_off;
  p.rope_cols = c.rope_cols; p.rope_period = c.rope_period; p.rope_offset = c.rope_offset;
  p.rope_ld = h->spec.max_positions;
  p.rope_cos = c.rope_period > 0 ? h->ptr<float>("rope.cos") : nullptr;
  p.rope_sin = c.rope_period > 0 ? h->ptr<float>("rope.sin") : nullptr;
  fill_norm_fields(h, c, p);
  const int m_tiles = (c.M + 2 * GEMM_BM - 1) / (2 * GEMM_BM), n_tiles = (c.N + BN - 1) / BN;
  const int pairs = std::min(m_tiles * n_tiles, h->num_sms / 2);
  const double valid_rows = c.grp_in == INT_MAX ? (double)c.M : (double)c.M / c.grp_in * c.grp_valid;
  const double out_bytes = valid_rows * c.N * (c.out_mode == OUT_BF16 ? 2.0 : (c.out_mode == OUT_F32 ? 4.0 : 8.0));
  McProfScope prof(h, 0, 2.0 * valid_rows * c.N * c.K, valid_rows * c.a_k_wrap * 2.0 + (double)c.N * c.K * 2.0 + out_bytes, stream);
  // specialised epilogues (gemm_sm100.cuh): TMA-store output, bias, whole 256-column tiles, rope on 64-wide heads
  const bool fast_ok = h->fast_epilogue && tma_out && c.bias != nullptr && c.N % BN == 0;
  if (norm_fast) return launch_gemm_pair_epi<EPI_RESID_NORM>(h, p, ma, mb, mo, mo2, pairs, stream);
  if (fast_ok && c.out_mode == OUT_BF16 && c.act == ACT_NONE && c.rope_period > 0 && c.rope_cols % 64 == 0)
    return launch_gemm_pair_epi<EPI_ROPE_BF16>(h, p, ma, mb, mo, mo2, pairs, stream);
  if (fast_ok && c.out_mode == OUT_BF16 && c.act == ACT_GELU_TANH && c.rope_period == 0)
    return launch_gemm_pair_epi<EPI_GELU_BF16>(h, p, ma, mb, mo, mo2, pairs, stream);
  if (fast_ok && c.out_mode == OUT_F32_RESIDUAL && c.act == ACT_NONE && c.rope_period == 0 && c.xb_out == nullptr)
    return launch_gemm_pair_epi<EPI_RESID_F32>(h, p, ma, mb, mo, mo2, pairs, stream);
  return launch_gemm_pair_epi<EPI_GENERIC>(h, p, ma, mb, mo, mo2, pairs, stream);
}

// Few-rows GEMM with K split over a cluster (gemm_splitk_sm100.cuh): S CTAs per 128 x 64 output tile.
template <int S>
int launch_gemm_splitk_s(mc_handle* h, const GemmCall& c, cudaStream_t stream) {
  constexpr int BN = 64;
  const CUtensorMap *ma, *mb;
  MC_TRY(get_map_2d_bf16(h, c.A, (uint64_t)c.a_k_wrap, (uint64_t)c.a_rows, GEMM_BK, GEMM_BM, &ma));
  MC_TRY(get_map_2d_bf16(h, c.W, (uint64_t)c.K, (uint64_t)c.N, GEMM_BK, BN, &mb));
  GemmParams p;
  p.tma_store = 0;
  p.M = c.M; p.N = c.N; p.K = c.K; p.a_k_wrap = c.a_k_wrap;
  p.bias = c.bias; p.act = c.act; p.out_mode = c.out_mode; p.out = c.out; p.ldo = c.ldo;
  p.grp_in = c.grp_in; p.grp_valid = c.grp_valid; p.grp_stride = c.grp_stride; p.grp_off = c.grp_off;
  p.rope_cols = c.rope_cols; p.rope_period = c.rope_period; p.rope_offset = c.rope_offset;
  p.rope_ld = h->spec.max_positions;
  p.rope_cos = c.rope_period > 0 ? h->ptr<float>("rope.cos") : nullptr;
  p.rope_sin = c.rope_period > 0 ? h->ptr<float>("rope.sin") : nullptr;
  if (h->l2_prefetch) { p.prefetch_ptr = c.prefetch_ptr; p.prefetch_bytes = c.prefetch_bytes; }
  fill_norm_fields(h, c, p);
  auto kernel = gemm_splitk_sm100_kernel<BN, S>;
  MC_TRY(mc_allow_smem(h, kernel, GemmSkCfg<BN>::kSmemBytes));
  const int m_tiles = (c.M + GEMM_BM - 1) / GEMM_BM, n_tiles = (c.N + BN - 1) / BN;
  const double valid_rows = c.grp_in == INT_MAX ? (double)c.M : (double)c.M / c.grp_in * c.grp_valid;
  const double out_bytes = valid_rows * c.N * (c.out_mode == OUT_BF16 ? 2.0 : (c.out_mode == OUT_F32 ? 4.0 : 8.0));
  McProfScope prof(h, 0, 2.0 * valid_rows * c.N * c.K, valid_rows * c.a_k_wrap * 2.0 + (double)c.N * c.K * 2.0 + out_bytes, stream);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(m_tiles * n_tiles * S); cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = GemmSkCfg<BN>::kSmemBytes; cfg.stream = stream;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = S; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = h->pdl ? 2 : 1;
  const int nkb = (c.K / GEMM_BK) / S;
  // k-blocks per barrier round trip: 1.  A CTA's slice is only 2 .. 10 k-blocks and the first MMA should start as soon as
  // the first k-block has landed; grouping them (measured: Wo 6.3 -> 6.7 us, W2 8.1 -> 8.6 us) delays it.
  const int kps = 1;
  (void)nkb;
  (void)cudaLaunchKernelEx(&cfg, kernel, *ma, *mb, p, kps);
  MC_LAUNCH_CHECK(h, "gemm_splitk_sm100_kernel");
  return MC_OK;
}

// S for a few-rows GEMM, or 0: the largest split (<= 8) that divides the k-blocks and keeps the grid within one CTA per
// SM.  Only GEMMs with few output tiles are split: measured in a dependent chain at M = 100 (tools/diag_small_gemm.py,
// profiles/r02_small_gemm_chain.log) Wo (16 tiles) goes 7.6 -> 6.3 us and W2 21.1 -> 8.1 us with S = 8, but QKV (48
// tiles) and W1 (64) are FASTER on the plain one-CTA-per-tile kernel (7.7 us) than split 4 ways (9.0 us): the cluster
// kernel's fixed cost (two cluster barriers, the DSMEM reduction at ~20 B/clk, two CTAs sharing an SM's tensor pipe)
// exceeds what their short K = 1024 loop can give back.
int pick_split_k(const mc_handle* h, const GemmCall& c) {
  if (c.M > 2 * GEMM_BM) return 0;
  const int base = ((c.M + GEMM_BM - 1) / GEMM_BM) * ((c.N + 63) / 64);
  const int num_kb = c.K / GEMM_BK;
  if (base > 32) {
    // a few more tiles, but a long K (the first transposed conv of the decoder: 40 tiles, K = 2048): two CTAs per SM
    if (base <= 48 && num_kb >= 32 && num_kb % 4 == 0) return 4;
    return 0;
  }
  for (int s = 8; s >= 2; s >>= 1)
    if (num_kb % s == 0 && num_kb / s >= 2 && base * s <= h->num_sms) return s;
  return 0;
}

int launch_gemm_splitk(mc_handle* h, const GemmCall& c, int S, cudaStream_t stream) {
  if (c.rope_period > 0 && c.rope_cols % 64 != 0) return h->fail(MC_ERR_ARG, "split-K gemm: rope needs 64-wide heads");
  if ((c.K / GEMM_BK) % S != 0) return h->fail(MC_ERR_ARG, "split-K gemm: %d k-blocks do not split %d ways", c.K / GEMM_BK, S);
  switch (S) {
    case 2: return launch_gemm_splitk_s<2>(h, c, stream);
    case 4: return launch_gemm_splitk_s<4>(h, c, stream);
    case 8: return launch_gemm_splitk_s<8>(h, c, stream);
    default: return h->fail(MC_ERR_ARG, "split-K gemm: unsupported split %d", S);
  }
}

int launch_gemm(mc_handle* h, const GemmCall& c, cudaStream_t stream) {
  if (c.K % GEMM_BK != 0 || c.K % c.a_k_wrap != 0 || c.a_k_wrap % GEMM_BK != 0)
    return h->fail(MC_ERR_ARG, "gemm: K=%d a_k_wrap=%d must be multiples of %d", c.K, c.a_k_wrap, GEMM_BK);
  if (c.N % 8 != 0) return h->fail(MC_ERR_ARG, "gemm: N=%d must be a multiple of 8", c.N);
  if (c.rope_period > 0 && c.rope_period + c.rope_offset > h->spec.max_positions)
    return h->fail(MC_ERR_ARG, "gemm: rope period %d exceeds table rows %d", c.rope_period, h->spec.max_positions);
  int bn = c.block_n;
  if (c.xb_out && (c.out_mode == OUT_BF16 || c.N % 64 != 0 || !c.xb_gamma || !c.stat_out))
    return h->fail(MC_ERR_ARG, "gemm: fused RMSNorm producer needs an fp32 output, N %% 64 == 0, gamma and a stats buffer");
  if (bn >= 1002 && bn <= 1008) return launch_gemm_splitk(h, c, bn - 1000, stream);   // forced (tests / A-B timing)
  if (bn == 4064 && (c.K / GEMM_BK) % 4 == 0) return launch_gemm_bn<64, GEMM_BM, 4>(h, c, stream);   // forced: 4 k-blocks per barrier round trip
  if (bn == 0 && (h->split_k == 2 || (h->split_k == 1 && h->in_session))) {
    const int S = pick_split_k(h, c);
    if (S >= 2) return launch_gemm_splitk(h, c, S, stream);
  }
  {
    // CTA pairs whenever there is at least one 256 x 256 tile per pair of SMs
    const int m2 = (c.M + 255) / 256, n2 = (c.N + 255) / 256;
    if ((bn == 0 && h->gemm_pair && c.N >= 256 && m2 * n2 >= h->num_sms / 2) || bn == 512) return launch_gemm_pair(h, c, stream);
  }
  if (bn == 0) {
    const int m_tiles = (c.M + GEMM_BM - 1) / GEMM_BM;
    if (c.N >= 256 && m_tiles * ((c.N + 255) / 256) >= 2 * h->num_sms) bn = 256;
    else if (c.N >= 128 && m_tiles * ((c.N + 127) / 128) >= h->num_sms) bn = 128;
    else if (c.N >= 256 && m_tiles * ((c.N + 255) / 256) >= h->num_sms) bn = 256;
    else bn = 64;
  }
  if (bn == 64 && c.block_n == 0 && (c.K / GEMM_BK) % 4 == 0 &&
      ((c.M + GEMM_BM - 1) / GEMM_BM) * ((c.N + 63) / 64) <= h->num_sms)
    return launch_gemm_bn<64, GEMM_BM, 4>(h, c, stream);   // one tile per CTA: four k-blocks per barrier round trip (bit-identical)
  switch (bn) {
    case 256: return launch_gemm_bn<256>(h, c, stream);
    case 128: return launch_gemm_bn<128>(h, c, stream);
    case 64: return launch_gemm_bn<64>(h, c, stream);
    default: return h->fail(MC_ERR_ARG, "gemm: unsupported block_n %d", bn);
  }
}

int ew_grid(mc_handle* h, long long work_items, int threads) {
  long long blocks = (work_items + threads - 1) / threads;
  const long long cap = (long long)h->num_sms * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

int launch_rmsnorm(mc_handle* h, const float* x, const float* gamma, bf16* out, int M, int d, int grp_in,
                   int64_t grp_stride, int64_t grp_off, cudaStream_t stream) {
  if (d % 4 != 0) return h->fail(MC_ERR_ARG, "rmsnorm: d=%d must be a multiple of 4", d);
  const int warps = 8;
  const int grid = ew_grid(h, M, warps);
  McProfScope prof(h, 3, 0.0, (double)M * d * 6.0, stream);
  const float eps = h->spec.norm_eps;
  switch (d % 128 == 0 ? d / 128 : 0) {   // register-resident rows (x read once) for the widths in use
    case 1: mc_launch(h, rmsnorm_rows_kernel<1>, dim3(grid), dim3(warps * 32), 0, stream, x, gamma, out, M, eps, grp_in, (long long)grp_stride, (long long)grp_off); break;
    case 2: mc_launch(h, rmsnorm_rows_kernel<2>, dim3(grid), dim3(warps * 32), 0, stream, x, gamma, out, M, eps, grp_in, (long long)grp_stride, (long long)grp_off); break;
    case 4: mc_launch(h, rmsnorm_rows_kernel<4>, dim3(grid), dim3(warps * 32), 0, stream, x, gamma, out, M, eps, grp_in, (long long)grp_stride, (long long)grp_off); break;
    case 8: mc_launch(h, rmsnorm_rows_kernel<8>, dim3(grid), dim3(warps * 32), 0, stream, x, gamma, out, M, eps, grp_in, (long long)grp_stride, (long long)grp_off); break;
    default: mc_launch(h, rmsnorm_kernel, dim3(grid), dim3(warps * 32), 0, stream, x, gamma, out, M, d, eps, grp_in, (long long)grp_stride, (long long)grp_off);
  }
  MC_LAUNCH_CHECK(h, "rmsnorm_kernel");
  return MC_OK;
}

// qkv [B*F, 3d] -> out [B*out_rows, d]: only the last out_rows queries of each window are kept.  phase (0 .. 15) places a
// window cut from a longer one on the key groups of the full-window pass (attn_sm100.cuh, ATTENTION CUTS); the SIMT
// kernel sums every row's keys from its own first key, so it is cut-invariant already and ignores it.
int launch_attention(mc_handle* h, const bf16* qkv, bf16* out, int B, int F, int out_rows, int phase, int impl, cudaStream_t stream) {
  if (out_rows < 1 || out_rows > F) return h->fail(MC_ERR_ARG, "attention: out_rows %d not in 1 .. %d", out_rows, F);
  const mc_spec& s = h->spec;
  const double span = std::min(F, s.window_left + s.window_right + 1);
  McProfScope prof(h, 1, 4.0 * B * out_rows * span * s.d_model,
                   (double)B * (F * 2.0 + out_rows * 2.0) * s.d_model * 2.0, stream);
  if (impl == 0 && attn_sm100_supported(s.window_left, s.window_right)) {   // v4 (P in tensor memory) or, with attn_p_tmem = 0, v3
    MC_TRY(launch_attention_sm100_v3(h, qkv, out, B, F, out_rows, phase, stream));
    return MC_OK;
  }
  if (impl != 0 && impl != 1) return h->fail(MC_ERR_ARG, "attention: unknown implementation %d (0 = tcgen05, 1 = SIMT cross-check)", impl);
  if (s.window_left + s.window_right + 1 > 160) return h->fail(MC_ERR_ARG, "attention window too wide");
  const long long warps = (long long)B * F * s.n_heads;
  const int threads = 256;
  const long long blocks = (warps * 32 + threads - 1) / threads;
  attention_window_simt_kernel<<<(unsigned)blocks, threads, 0, stream>>>(qkv, out, B, F, s.n_heads, s.window_left,
                                                                         s.window_right, out_rows, 0.125f);
  MC_LAUNCH_CHECK(h, "attention_window_simt_kernel");
  return MC_OK;
}

// ------------------------------------------------------- transformer stack
struct StackBufs {
  float* x;   // [M,d] fp32 residual stream
  float* x2;  // [M,d] second residual buffer (row compaction between layers ping-pongs x <-> x2)
  bf16* hbuf; // [M,d]
  bf16* qkv;  // [M,3d]
  bf16* att;  // [M,d]
  bf16* ffn;  // [M,f]
  float* stats;  // [M, d/64] per-row partial sums of x^2 (fused RMSNorm on the few-rows path)
};

// RMSNorm folded into the neighbouring GEMMs (GemmParams: producer / consumer): only on the few-rows path, i.e. under the
// same switch as the split-K kernels, so that a session and a stateless call in the same mode run identical kernels.
bool few_rows_regime(const mc_handle* h, long long M) {
  return (h->split_k == 2 || (h->split_k == 1 && h->in_session)) && M <= 2 * GEMM_BM;
}
// fuse_norm: 0 never; 1 few-rows path only (default); 2 every size, Wo and W2 produce; 3 every size, only Wo produces
// (norm1 stays a kernel) — 2 / 3 are the offline variants measured in DESIGN.md §8.
bool fuse_norm_ok(const mc_handle* h, long long M) {
  if (h->spec.d_model % 64 != 0 || h->fuse_norm == 0) return false;
  return h->fuse_norm >= 2 || few_rows_regime(h, M);
}

// x [M, d] -> b.hbuf = bf16(x * gamma), b.stats: the first producer of a fused stack when no GEMM can play that role
int launch_rowstats(mc_handle* h, const float* x, const float* gamma, bf16* xb, float* stats, long long M, int d, cudaStream_t stream) {
  McProfScope prof(h, 3, 0.0, (double)M * d * 6.0, stream);
  mc_launch(h, rowstats_cast_kernel, dim3(ew_grid(h, M * (d / 64), 256)), dim3(256), 0, stream, x, gamma, xb, stats, M, d);
  MC_LAUNCH_CHECK(h, "rowstats_cast_kernel");
  return MC_OK;
}

// Runs n_layers blocks over B windows of F frames held in b.x and returns, in *x_out, the residual
// stream restricted to the LAST keep_rows frames of every window ([B*keep_rows, d]).
//
// Dead-output elimination (exact): a layer whose output is needed only for the last R_out rows
// needs keys/values for the last R_in = min(F, R_out + window_left) rows, so working backwards from
// keep_rows each layer gets (R_in, R_out); rows outside are never computed.  Per-row arithmetic is
// unchanged (same K order, same epilogues), and attention lays a cut window out on the full pass's
// 16-key groups (phase = (F - R_in) mod 16, attn_sm100.cuh), so kept rows are bit-identical to the full pass.
//
// fused = true (few-rows path): the caller has already put bf16(x * gamma_norm1[0]) in b.hbuf and the rows' partial sums
// of squares in b.stats (its last GEMM ran as a "producer"); every norm of the stack then lives in GEMM epilogues — QKV
// and W1 scale their accumulator rows by rs(row), Wo and W2 emit the next norm's operand — and no rmsnorm kernel is
// launched.  final_gamma (may be NULL) is the weight of the norm that FOLLOWS the stack: the last W2 emits that
// operand, returned with its statistics through xb_out / stats_out.
int run_layers(mc_handle* h, const char* prefix, int n_layers, const StackBufs& b, int B, int F, int keep_rows,
               float** x_out, cudaStream_t stream, int fuse_mode = 0 /* 0 none, 1 every norm, 2 only norm2 (Wo -> W1) */,
               const float* final_gamma = nullptr, bf16** xb_out = nullptr, float** stats_out = nullptr) {
  const mc_spec& s = h->spec;
  const int d = s.d_model, f = s.ffn_dim;
  const int nst = d / 64;
  const bool fused = fuse_mode == 1;        // norm1 in (W2 | first producer) -> QKV
  const bool fused2 = fuse_mode != 0;       // norm2 in Wo -> W1
  std::vector<int> r_in(n_layers), r_out(n_layers);
  {
    int need = std::max(1, std::min(keep_rows, F));
    // One 128-row tile (a batch-1 streaming pass): dropping rows saves nothing — every GEMM is one tile either way —
    // and the row compactions would be three more launches on the latency path.  Per-row results do not depend on
    // which other rows are computed, so this stays bit-identical.
    if (B == 1 && F <= GEMM_BM) need = F;
    for (int l = n_layers - 1; l >= 0; --l) {
      r_out[l] = need;
      need = (need >= F) ? F : std::min(F, need + s.window_left);
      // exact_cut = 0: the earlier plan, which cut windows only at multiples of 16 frames (kept for A/B runs)
      if (!h->exact_cut && need < F) need = F - ((F - need) / 16) * 16;
      r_in[l] = need;
    }
  }
  float* x = b.x;
  float* xalt = b.x2;
  int rows = F;  // rows per window currently held in x
  char name[128];
  for (int l = 0; l < n_layers; ++l) {
    auto T = [&](const char* leaf) {
      snprintf(name, sizeof(name), "%s.layers.%d.%s", prefix, l, leaf);
      return std::string(name);
    };
    const int Ri = rows, Ro = std::min(r_out[l], rows);
    const int Mi = B * Ri, Mo = B * Ro;
    if (!fused) MC_TRY(launch_rmsnorm(h, x, h->ptr<float>(T("norm1")), b.hbuf, Mi, d, INT_MAX, 0, 0, stream));
    GemmCall g{};
    if (fused) { g.row_stats = b.stats; g.row_stats_n = nst; }
    g.A = b.hbuf; g.a_rows = Mi; g.a_k_wrap = d; g.W = h->ptr<bf16>(T("wqkv")); g.bias = h->ptr<float>(T("bqkv"));
    g.M = Mi; g.N = 3 * d; g.K = d; g.act = ACT_NONE; g.out_mode = OUT_BF16; g.out = b.qkv; g.ldo = 3 * d;
    g.rope_cols = 2 * d; g.rope_period = Ri; g.rope_offset = F - Ri;
    g.prefetch_ptr = h->ptr<bf16>(T("wo")); g.prefetch_bytes = (long long)d * d * 2;
    MC_TRY(launch_gemm(h, g, stream));
    MC_TRY(launch_attention(h, b.qkv, b.att, B, Ri, Ro, (F - Ri) % 16, h->attn_impl, stream));
    if (Ro < Ri) {
      const long long items = (long long)Mo * (d / 4);
      McProfScope prof(h, 3, 0.0, (double)Mo * d * 8.0, stream);
      mc_launch(h, compact_rows_kernel, dim3(ew_grid(h, items, 256)), dim3(256), 0, stream, reinterpret_cast<const float4*>(x),
                reinterpret_cast<float4*>(xalt), B, Ri, Ro, d / 4);
      MC_LAUNCH_CHECK(h, "compact_rows_kernel");
      std::swap(x, xalt);
      rows = Ro;
    }
    GemmCall o{};
    o.A = b.att; o.a_rows = Mo; o.a_k_wrap = d; o.W = h->ptr<bf16>(T("wo")); o.bias = h->ptr<float>(T("bo"));
    o.M = Mo; o.N = d; o.K = d; o.act = ACT_NONE; o.out_mode = OUT_F32_RESIDUAL; o.out = x; o.ldo = d;
    o.prefetch_ptr = h->ptr<bf16>(T("w1")); o.prefetch_bytes = (long long)f * d * 2;
    if (fused2) { o.xb_out = b.hbuf; o.xb_gamma = h->ptr<float>(T("norm2")); o.stat_out = b.stats; }
    MC_TRY(launch_gemm(h, o, stream));
    if (!fused2) MC_TRY(launch_rmsnorm(h, x, h->ptr<float>(T("norm2")), b.hbuf, Mo, d, INT_MAX, 0, 0, stream));
    GemmCall u{};
    if (fused2) { u.row_stats = b.stats; u.row_stats_n = nst; }
    u.A = b.hbuf; u.a_rows = Mo; u.a_k_wrap = d; u.W = h->ptr<bf16>(T("w1")); u.bias = h->ptr<float>(T("b1"));
    u.M = Mo; u.N = f; u.K = d; u.act = ACT_GELU_TANH; u.out_mode = OUT_BF16; u.out = b.ffn; u.ldo = f;
    u.prefetch_ptr = h->ptr<bf16>(T("w2")); u.prefetch_bytes = (long long)d * f * 2;
    MC_TRY(launch_gemm(h, u, stream));
    GemmCall w{};
    w.A = b.ffn; w.a_rows = Mo; w.a_k_wrap = f; w.W = h->ptr<bf16>(T("w2")); w.bias = h->ptr<float>(T("b2"));
    w.M = Mo; w.N = d; w.K = f; w.act = ACT_NONE; w.out_mode = OUT_F32_RESIDUAL; w.out = x; w.ldo = d;
    if (l + 1 < n_layers) {
      snprintf(name, sizeof(name), "%s.layers.%d.wqkv", prefix, l + 1);
      w.prefetch_ptr = h->ptr<bf16>(name); w.prefetch_bytes = (long long)3 * d * d * 2;
    }
    if (fused) {
      const float* next_gamma = final_gamma;
      if (l + 1 < n_layers) {
        snprintf(name, sizeof(name), "%s.layers.%d.norm1", prefix, l + 1);
        next_gamma = h->ptr<float>(name);
      }
      if (next_gamma) { w.xb_out = b.hbuf; w.xb_gamma = next_gamma; w.stat_out = b.stats; }
    }
    MC_TRY(launch_gemm(h, w, stream));
  }
  bf16* xb = b.hbuf;
  float* st = b.stats;
  if (rows > keep_rows && B == 1) {
    x += (size_t)(rows - keep_rows) * d;   // one window: its last rows are already contiguous — no copy
    xb += (size_t)(rows - keep_rows) * d;
    st += (size_t)(rows - keep_rows) * nst;
  } else if (rows > keep_rows) {  // single-tile passes keep every row through the layers: compact at the end
    const int Ro = keep_rows;
    const long long items = (long long)B * Ro * (d / 4);
    mc_launch(h, compact_rows_kernel, dim3(ew_grid(h, items, 256)), dim3(256), 0, stream, reinterpret_cast<const float4*>(x),
              reinterpret_cast<float4*>(xalt), B, rows, Ro, d / 4);
    MC_LAUNCH_CHECK(h, "compact_rows_kernel");
    std::swap(x, xalt);
  }
  if (fused && final_gamma && rows > keep_rows && B != 1) return h->fail(MC_ERR_STATE, "run_layers: fused norms with a trailing compaction");
  *x_out = x;
  if (xb_out) *xb_out = xb;
  if (stats_out) *stats_out = st;
  return MC_OK;
}

StackBufs carve_stack(Carver& cv, uint8_t* base, int M, int d, int f, bool dry) {
  StackBufs b{};
  size_t ox = cv.take((size_t)M * d * 4), ox2 = cv.take((size_t)M * d * 4), oh = cv.take((size_t)M * d * 2),
         oq = cv.take((size_t)M * 3 * d * 2), oa = cv.take((size_t)M * d * 2), of = cv.take((size_t)M * f * 2),
         os = cv.take((size_t)M * (d / 64 + 1) * 4);
  if (!dry) {
    b.stats = reinterpret_cast<float*>(base + os);
    b.x = reinterpret_cast<float*>(base + ox);
    b.x2 = reinterpret_cast<float*>(base + ox2);
    b.hbuf = reinterpret_cast<bf16*>(base + oh);
    b.qkv = reinterpret_cast<bf16*>(base + oq);
    b.att = reinterpret_cast<bf16*>(base + oa);
    b.ffn = reinterpret_cast<bf16*>(base + of);
  }
  return b;
}

int launch_vq(mc_handle* h, const float* z, int n_items, int F, int keep, int64_t* codes, float* margin,
              void* scratch, cudaStream_t stream);
size_t vq_scratch_bytes(mc_handle* h, int Mq);

// ----------------------------------------------------------------- encode
// Encoder conv stack over Bc items of Tc samples (item b at wav + b*ld; samples >= Tc read as zero): conv0 on CUDA
// cores, the rest as implicit GEMMs.  The last conv writes fp32 rows [Tc/hop, d] per item at x_out + b*x_item_stride.
struct ConvPlan {
  int B = 0, T = 0;
  std::vector<int> Tl;          // output length of every conv
  std::vector<size_t> off;      // workspace offset of the (left-padded) bf16 output of conv i, i < n-1
};

ConvPlan plan_conv(const mc_spec& s, Carver& cv, int Bc, int Tc_padded) {
  ConvPlan p;
  p.B = Bc; p.T = Tc_padded;
  const int n = s.n_convs;
  p.Tl.resize(n); p.off.resize(n);
  int t = Tc_padded;
  for (int i = 0; i < n; ++i) { t /= s.conv_strides[i]; p.Tl[i] = t; }
  for (int i = 0; i + 1 < n; ++i)
    p.off[i] = cv.take((size_t)Bc * (s.conv_strides[i + 1] + p.Tl[i]) * s.conv_channels[i] * 2 + 65536);
  return p;
}

int run_conv_stack(mc_handle* h, const ConvPlan& cp, uint8_t* base, const float* wav, int64_t ld, int Tvalid,
                   float* x_out, int64_t x_item_stride, cudaStream_t stream, bf16* xb_out = nullptr,
                   const float* xb_gamma = nullptr, float* stat_out = nullptr) {
  const mc_spec& s = h->spec;
  const int n = s.n_convs, d = s.d_model, B = cp.B;
  const std::vector<int>& Tl = cp.Tl;
  const int* Cl = s.conv_channels;
  {  // zero the left padding of every conv input (one launch)
    PadList pl;
    long long work = 0;
    for (int i = 0; i + 1 < n; ++i) {
      const int pad = s.conv_strides[i + 1];
      pl.base[pl.n] = base + cp.off[i];
      pl.pitch[pl.n] = (long long)(pad + Tl[i]) * Cl[i] * 2;
      pl.width[pl.n] = pad * Cl[i] * 2;
      if (pl.width[pl.n] % 16 != 0 || pl.pitch[pl.n] % 16 != 0) return h->fail(MC_ERR_ARG, "conv %d: padding is not 16-byte granular", i + 1);
      work = std::max(work, (long long)B * (pl.width[pl.n] >> 4));
      ++pl.n;
    }
    if (pl.n > 0) {
      mc_launch(h, zero_pads_kernel, dim3(ew_grid(h, work, 256)), dim3(256), 0, stream, pl, B);
      MC_LAUNCH_CHECK(h, "zero_pads_kernel");
    }
  }
  {
    const int s0 = s.conv_strides[0], C0 = Cl[0];
    const int cgroups = C0 / 8;
    if ((2 * s0 != 8 && 2 * s0 != 16) || C0 % 8 != 0 || 256 % cgroups != 0)
      return h->fail(MC_ERR_ARG, "conv0: stride %d / channels %d unsupported", s0, C0);
    const int threads = 256;
    const long long frames = (long long)B * Tl[0];
    const int grid = ew_grid(h, frames * cgroups, threads);
    McProfScope prof(h, 3, 2.0 * B * Tl[0] * 2 * s0 * C0, (double)B * Tvalid * 4.0 + (double)B * Tl[0] * C0 * 2.0, stream);
    bf16* o0 = reinterpret_cast<bf16*>(base + cp.off[0]);
    if (2 * s0 == 8)
      mc_launch(h, conv_first_kernel<8>, dim3(grid), dim3(threads), 0, stream, wav, (long long)ld, Tvalid, B, Tl[0], s0, C0,
                h->ptr<float>("enc.conv0.w"), h->ptr<float>("enc.conv0.b"), o0, (int)s.conv_strides[1]);
    else
      mc_launch(h, conv_first_kernel<16>, dim3(grid), dim3(threads), 0, stream, wav, (long long)ld, Tvalid, B, Tl[0], s0, C0,
                h->ptr<float>("enc.conv0.w"), h->ptr<float>("enc.conv0.b"), o0, (int)s.conv_strides[1]);
    MC_LAUNCH_CHECK(h, "conv_first_kernel");
  }
  for (int i = 1; i < n; ++i) {
    const int si = s.conv_strides[i];
    const long long rows = (long long)B * (1 + Tl[i]);
    if (rows > INT_MAX) return h->fail(MC_ERR_ARG, "encode: conv %d has too many rows", i);
    GemmCall g{};
    g.A = reinterpret_cast<const bf16*>(base + cp.off[i - 1]);
    g.a_k_wrap = si * Cl[i - 1];
    g.a_rows = rows;
    g.W = h->ptr<bf16>("enc.conv" + std::to_string(i) + ".w");
    g.bias = h->ptr<float>("enc.conv" + std::to_string(i) + ".b");
    g.M = (int)rows; g.N = Cl[i]; g.K = 2 * g.a_k_wrap;
    g.grp_in = 1 + Tl[i]; g.grp_valid = Tl[i];
    if (i + 1 < n) {
      const int pad = s.conv_strides[i + 1];
      g.act = ACT_GELU_TANH; g.out_mode = OUT_BF16; g.out = base + cp.off[i]; g.ldo = Cl[i];
      g.grp_stride = (int64_t)(pad + Tl[i]) * Cl[i]; g.grp_off = (int64_t)pad * Cl[i];
    } else {
      g.act = ACT_NONE; g.out_mode = OUT_F32; g.out = x_out; g.ldo = d;
      g.grp_stride = x_item_stride; g.grp_off = 0;
      g.xb_out = xb_out; g.xb_gamma = xb_gamma; g.stat_out = stat_out;   // fused RMSNorm: first producer of the encoder stack
    }
    MC_TRY(launch_gemm(h, g, stream));
  }
  return MC_OK;
}

// Frames of the conv stem whose value can depend on where a window starts: the causal convs see zeros
// instead of real history only through a chain of "first output" positions, which ends after frame 1
// (checked layer by layer for the strides in the spec; see DESIGN.md §4 "shared convolution stem").
int stem_prefix_frames(const mc_spec& s) {
  // a conv output at position v is window-specific iff one of its inputs [v*st - st, v*st + st) is padding or
  // window-specific; `dirty` = number of leading window-specific positions at the current level
  long long dirty = 0;   // raw samples: none are window-specific, only the padding is
  for (int i = 0; i < s.n_convs; ++i) {
    const int st = s.conv_strides[i];
    // position v reads inputs up to... it is clean iff v*st - st >= dirty  <=>  v >= dirty/st + 1 (ceil)
    dirty = (dirty + st - 1) / st + 1;
  }
  return (int)dirty;
}

// Frames a decode cut from a longer window needs before its first kept sample.  Transposed conv i (stride ds[i]) reads
// input steps t−1 and t, so the zero left pad of a cut window spoils its first ds[i] outputs, and the spoiled prefix
// grows through the stack to L = Σ_i hop / Π_{j<i} ds[j] samples (404 for strides (4, 4, 4, 5)).  The margin is
// ceil(L / hop): 2 frames for the default strides, more when a late encoder stride is small (3 for (4, 4, 5, 1)).
int tconv_margin_frames(const mc_spec& s) {
  const int n = s.n_convs;
  int hop = 1;
  for (int i = 0; i < n; ++i) hop *= s.conv_strides[i];
  long long look_back = 0, step = hop;   // step: samples per input position of decoder conv i
  for (int i = 0; i < n; ++i) {
    look_back += step;
    step /= s.conv_strides[n - 1 - i];
  }
  return (int)((look_back + hop - 1) / hop);
}

// A ragged session-pool batch (mc_pool_push_audio_ragged): encode_impl's `keep` rows of every window run through the
// stack, then each item's own last `keep` frames (rtable: pool_roll_ragged_kernel's table) are gathered for the VQ.
struct RaggedKeep {
  const int* rtable;
  int C, keep;
};

int encode_impl(mc_handle* h, const float* wav, int64_t ld, int B, int T, int keep, int64_t* codes, float* margin,
                float* z_e_out, cudaStream_t stream, const RaggedKeep* ragged = nullptr) {
  const mc_spec& s = h->spec;
  const int n = s.n_convs;
  int hop = 1;
  for (int i = 0; i < n; ++i) hop *= s.conv_strides[i];
  const int F = (T + hop - 1) / hop;
  if (F < 1) return h->fail(MC_ERR_ARG, "encode: empty input");
  if (F > s.max_positions) return h->fail(MC_ERR_ARG, "encode: %d frames exceed RoPE table (%d rows)", F, s.max_positions);
  if (keep <= 0 || keep > F) keep = F;
  const int Tp = F * hop;
  const int d = s.d_model, dq = s.codebook_dim;
  const long long Mll = (long long)B * F;
  if (Mll * std::max(3 * d, s.ffn_dim) > (long long)INT_MAX) return h->fail(MC_ERR_ARG, "encode: batch too large");
  const int M = (int)Mll;

  // Shared convolution stem (exact): overlapping windows whose starts are hop-aligned see identical conv
  // outputs from frame `pre` on, so the stack runs ONCE over the whole span and per window only over the
  // first `pre` frames; the windows' residual streams are then gathered from the span's frames.
  const int pre = stem_prefix_frames(s);
  const long long span_samples = (long long)(B - 1) * ld + T;
  const long long span_frames = span_samples / hop;
  const bool shared = h->shared_stem && B >= 2 && ld > 0 && ld < T && ld % hop == 0 && T % hop == 0 && F > pre &&
                      span_samples <= INT_MAX && span_frames + (long long)pre * B < (long long)B * F / 2;
  // RMSNorms inside GEMM epilogues on the few-rows path (the keep < F case with several windows compacts rows at the end)
  // RMSNorms in GEMM epilogues.  Few-rows regime: the last conv GEMM itself is the first producer (+ B: it carries one junk
  // row per window); otherwise one rowstats pass after the conv stack.
  const int fuse_mode = !(fuse_norm_ok(h, Mll + B) && s.enc_layers > 0) ? 0 : ((h->fuse_norm == 3 && !few_rows_regime(h, Mll + B)) ? 2 : 1);
  const bool fused = fuse_mode == 1;
  const bool conv_producer = fused && few_rows_regime(h, Mll + B) && !shared;

  // ---- carve workspace (sizes first, then pointers)
  Carver cv;
  ConvPlan cp_full, cp_span, cp_pre;
  size_t ostem = 0;
  if (shared) {
    cp_span = plan_conv(s, cv, 1, (int)span_samples);
    cp_pre = plan_conv(s, cv, B, pre * hop);
    ostem = cv.take((size_t)span_frames * d * 4);
  } else {
    cp_full = plan_conv(s, cv, B, Tp);
  }
  Carver cv2 = cv;
  carve_stack(cv2, nullptr, M, d, s.ffn_dim, true);
  size_t oz = cv2.take((size_t)M * dq * 4);
  size_t ovq = cv2.take(vq_scratch_bytes(h, B * keep));
  const size_t ozg = ragged ? cv2.take((size_t)B * ragged->keep * dq * 4) : 0;
  MC_TRY(arena_reserve(h, cv2.off, stream));
  uint8_t* base = h->arena;
  StackBufs sb = carve_stack(cv, base, M, d, s.ffn_dim, false);
  float* z_e = reinterpret_cast<float*>(base + oz);
  void* vq_scratch = base + ovq;

  // ---- conv stack -> fp32 residual stream sb.x [B*F, d]
  if (shared) {
    float* stem = reinterpret_cast<float*>(base + ostem);
    MC_TRY(run_conv_stack(h, cp_span, base, wav, span_samples, (int)span_samples, stem, 0, stream));
    MC_TRY(run_conv_stack(h, cp_pre, base, wav, ld, pre * hop, sb.x, (int64_t)F * d, stream));
    const long long items = (long long)B * (F - pre) * (d / 4);
    McProfScope prof(h, 3, 0.0, (double)B * (F - pre) * d * 8.0, stream);
    mc_launch(h, gather_stem_kernel, dim3(ew_grid(h, items, 256)), dim3(256), 0, stream, reinterpret_cast<const float4*>(stem),
              reinterpret_cast<float4*>(sb.x), B, F, pre, (int)(ld / hop), d / 4);
    MC_LAUNCH_CHECK(h, "gather_stem_kernel");
  } else {
    if (conv_producer)
      MC_TRY(run_conv_stack(h, cp_full, base, wav, ld, T, sb.x, (int64_t)F * d, stream, sb.hbuf, h->ptr<float>("enc.layers.0.norm1"), sb.stats));
    else
      MC_TRY(run_conv_stack(h, cp_full, base, wav, ld, T, sb.x, (int64_t)F * d, stream));
  }
  if (fused && !conv_producer) MC_TRY(launch_rowstats(h, sb.x, h->ptr<float>("enc.layers.0.norm1"), sb.hbuf, sb.stats, M, d, stream));
  // ---- transformer (only the rows the kept frames depend on, unless the full latents are requested)
  const int keep_rows = z_e_out ? F : keep;
  float* xk = nullptr;
  bf16* xbk = sb.hbuf;
  float* stk = nullptr;
  MC_TRY(run_layers(h, "enc", s.enc_layers, sb, B, F, keep_rows, &xk, stream, fuse_mode, fused ? h->ptr<float>("enc.norm_f") : nullptr, &xbk, &stk));
  const int Mk = B * keep_rows;
  if (!fused) MC_TRY(launch_rmsnorm(h, xk, h->ptr<float>("enc.norm_f"), sb.hbuf, Mk, d, INT_MAX, 0, 0, stream));
  GemmCall pj{};
  if (fused) { pj.row_stats = stk; pj.row_stats_n = d / 64; }
  pj.A = fused ? xbk : sb.hbuf; pj.a_rows = Mk; pj.a_k_wrap = d; pj.W = h->ptr<bf16>("enc.proj.w"); pj.bias = h->ptr<float>("enc.proj.b");
  pj.M = Mk; pj.N = dq; pj.K = d; pj.act = ACT_NONE; pj.out_mode = OUT_F32; pj.out = z_e; pj.ldo = dq;
  MC_TRY(launch_gemm(h, pj, stream));
  if (z_e_out) MC_CUDA(h, cudaMemcpyAsync(z_e_out, z_e, (size_t)M * dq * 4, cudaMemcpyDeviceToDevice, stream));
  // ---- quantise the kept frames (z_e holds keep_rows rows per window)
  if (ragged) {
    float* zg = reinterpret_cast<float*>(base + ozg);
    pool_gather_rows_ragged_kernel<<<dim3(1, B), 256, 0, stream>>>(z_e, ragged->rtable, ragged->C, keep_rows, F, ragged->keep,
                                                                   dq, hop, zg);
    MC_LAUNCH_CHECK(h, "pool_gather_rows_ragged_kernel");
    return launch_vq(h, zg, B, ragged->keep, ragged->keep, codes, margin, vq_scratch, stream);
  }
  MC_TRY(launch_vq(h, z_e, B, keep_rows, keep, codes, margin, vq_scratch, stream));
  return MC_OK;
}

// ----------------------------------------------------------------- decode
int decode_impl(mc_handle* h, const int64_t* codes, const float* z_q, int B, int F, int keep, float* wav,
                cudaStream_t stream) {
  const mc_spec& s = h->spec;
  const int n = s.n_convs;
  if (F < 1 || B < 1) return h->fail(MC_ERR_ARG, "decode: empty input");
  if (F > s.max_positions) return h->fail(MC_ERR_ARG, "decode: %d frames exceed RoPE table (%d rows)", F, s.max_positions);
  int hop = 1;
  for (int i = 0; i < n; ++i) hop *= s.conv_strides[i];
  const int d = s.d_model;
  const long long Mll = (long long)B * F;
  if (Mll * std::max(3 * d, s.ffn_dim) > (long long)INT_MAX) return h->fail(MC_ERR_ARG, "decode: batch too large");
  const int M = (int)Mll;
  const int total = F * hop;
  if (keep <= 0 || keep > total) keep = total;
  // decoder conv i: channels dch[i] -> dch[i+1], stride ds[i]; input length Tin[i]
  std::vector<int> dch(n + 1), ds(n), Tin(n);
  dch[0] = d;
  for (int i = 0; i < n; ++i) {
    ds[i] = s.conv_strides[n - 1 - i];
    dch[i + 1] = (n - 2 - i >= 0) ? s.conv_channels[n - 2 - i] : 1;
  }
  // Frames whose samples are kept, plus the margin the causal transposed convs look back over (tconv_margin_frames).
  const int Rk = (keep >= total) ? F : std::min(F, (keep + hop - 1) / hop + tconv_margin_frames(s));
  Tin[0] = Rk;
  for (int i = 1; i < n; ++i) Tin[i] = Tin[i - 1] * ds[i - 1];

  Carver cv;
  size_t oa0 = cv.take((size_t)M * 64 * 2);
  std::vector<size_t> tb_off(n);
  for (int i = 0; i < n; ++i) tb_off[i] = cv.take((size_t)B * (1 + Tin[i]) * dch[i] * 2 + 65536);
  Carver cv2 = cv;
  carve_stack(cv2, nullptr, M, d, s.ffn_dim, true);
  MC_TRY(arena_reserve(h, cv2.off, stream));
  uint8_t* base = h->arena;
  StackBufs sb = carve_stack(cv, base, M, d, s.ffn_dim, false);
  bf16* a0 = reinterpret_cast<bf16*>(base + oa0);

  const int threads = 256;
  if (codes) {
    mc_launch(h, embed_codes_kernel, dim3(ew_grid(h, (long long)M * 8, threads)), dim3(threads), 0, stream,
              reinterpret_cast<const long long*>(codes), h->ptr<float>("vq.codebook"), (int)s.codebook_size, a0, (long long)M);
    MC_LAUNCH_CHECK(h, "embed_codes_kernel");
  } else {
    pack_latents_kernel<<<ew_grid(h, (long long)M * 8, threads), threads, 0, stream>>>(z_q, a0, M);
    MC_LAUNCH_CHECK(h, "pack_latents_kernel");
  }
  GemmCall ip{};
  ip.A = a0; ip.a_rows = M; ip.a_k_wrap = 64; ip.W = h->ptr<bf16>("dec.in_proj.w"); ip.bias = h->ptr<float>("dec.in_proj.b");
  ip.M = M; ip.N = d; ip.K = 64; ip.act = ACT_NONE; ip.out_mode = OUT_F32; ip.out = sb.x; ip.ldo = d;
  const int fuse_mode = !(fuse_norm_ok(h, Mll) && s.dec_layers > 0) ? 0 : ((h->fuse_norm == 3 && !few_rows_regime(h, Mll)) ? 2 : 1);
  const bool fused = fuse_mode == 1;
  const bool proj_producer = fused && few_rows_regime(h, Mll);
  if (proj_producer) { ip.xb_out = sb.hbuf; ip.xb_gamma = h->ptr<float>("dec.layers.0.norm1"); ip.stat_out = sb.stats; }
  MC_TRY(launch_gemm(h, ip, stream));
  if (fused && !proj_producer) MC_TRY(launch_rowstats(h, sb.x, h->ptr<float>("dec.layers.0.norm1"), sb.hbuf, sb.stats, M, d, stream));
  float* xk = nullptr;
  MC_TRY(run_layers(h, "dec", s.dec_layers, sb, B, F, Rk, &xk, stream, fuse_mode));

  {  // zero row 0 (left pad) of every transposed-conv input (one launch)
    PadList pl;
    long long work = 0;
    for (int i = 0; i < n; ++i) {
      pl.base[pl.n] = base + tb_off[i];
      pl.pitch[pl.n] = (long long)(1 + Tin[i]) * dch[i] * 2;
      pl.width[pl.n] = dch[i] * 2;
      if (pl.width[pl.n] % 16 != 0) return h->fail(MC_ERR_ARG, "tconv %d: %d channels are not 16-byte granular", i, dch[i]);
      work = std::max(work, (long long)B * (pl.width[pl.n] >> 4));
      ++pl.n;
    }
    mc_launch(h, zero_pads_kernel, dim3(ew_grid(h, work, 256)), dim3(256), 0, stream, pl, B);
    MC_LAUNCH_CHECK(h, "zero_pads_kernel");
  }
  MC_TRY(launch_rmsnorm(h, xk, h->ptr<float>("dec.norm_f"), reinterpret_cast<bf16*>(base + tb_off[0]), B * Rk, d, Rk,
                        (int64_t)(1 + Rk) * d, d, stream));
  for (int i = 0; i + 1 < n; ++i) {
    GemmCall g{};
    g.A = reinterpret_cast<const bf16*>(base + tb_off[i]);
    g.a_k_wrap = dch[i]; g.a_rows = (int64_t)B * (1 + Tin[i]);
    g.W = h->ptr<bf16>("dec.up" + std::to_string(i) + ".w");
    g.bias = h->ptr<float>("dec.up" + std::to_string(i) + ".b");
    g.M = B * (1 + Tin[i]); g.N = ds[i] * dch[i + 1]; g.K = 2 * dch[i];
    g.grp_in = 1 + Tin[i]; g.grp_valid = Tin[i];
    g.act = ACT_GELU_TANH; g.out_mode = OUT_BF16; g.out = base + tb_off[i + 1]; g.ldo = g.N;
    g.grp_stride = (int64_t)(1 + Tin[i + 1]) * dch[i + 1]; g.grp_off = dch[i + 1];
    MC_TRY(launch_gemm(h, g, stream));
  }
  {
    const int i = n - 1;
    if (ds[i] > 8 || dch[i] % 8 != 0) return h->fail(MC_ERR_ARG, "last tconv: stride %d / channels %d unsupported", ds[i], dch[i]);
    const long long items = (long long)B * Tin[i];
    const size_t smem = (size_t)dch[i] * 2 * ds[i] * 4;
    // the weight table outgrows the default 48 KB from Cin * stride > 6144 on (e.g. 1024 channels at stride 8); the
    // attribute is per function, so it is raised to the largest table a spec can ask for (2048 channels, stride 8)
    if (smem > 48 * 1024) MC_TRY(mc_allow_smem(h, tconv_last_kernel<8>, 2048 * 2 * 8 * 4));
    McProfScope prof(h, 3, 4.0 * B * Tin[i] * dch[i] * ds[i], (double)B * Tin[i] * dch[i] * 2.0 + (double)B * keep * 4.0, stream);
    mc_launch(h, tconv_last_kernel<8>, dim3(ew_grid(h, items, threads)), dim3(threads), smem, stream,
              reinterpret_cast<const bf16*>(base + tb_off[i]), B, Tin[i], dch[i], ds[i],
              h->ptr<float>("dec.up" + std::to_string(i) + ".w"), h->ptr<float>("dec.up" + std::to_string(i) + ".b"), wav, keep);
    MC_LAUNCH_CHECK(h, "tconv_last_kernel");
  }
  return MC_OK;
}

// --------------------------------------------------------------------- VQ
size_t vq_scratch_bytes(mc_handle* h, int Mq) {
  return std::max(vq_sm100_scratch_bytes(h->num_sms, Mq), (size_t)64 * Mq * sizeof(VqPartial)) + 1024;
}

int launch_vq(mc_handle* h, const float* z, int n_items, int F, int keep, int64_t* codes, float* margin,
              void* scratch, cudaStream_t stream) {
  const mc_spec& s = h->spec;
  const int Mq = n_items * keep;
  McProfScope prof(h, 2, 2.0 * Mq * (double)s.codebook_size * s.codebook_dim, (double)s.codebook_size * 128.0, stream);
  if (h->vq_impl == 0) {
    return launch_vq_sm100(h, z, n_items, F, keep, codes, margin, scratch, stream);
  }
  const int row_tiles = (Mq + 127) / 128;
  int splits = (2 * h->num_sms + row_tiles - 1) / row_tiles;
  splits = std::max(1, std::min(64, splits));
  vq_simt_kernel<<<dim3(row_tiles, splits), 128, 0, stream>>>(z, Mq, F, keep, h->ptr<float>("vq.codebook"),
                                                              h->ptr<float>("vq.c2"), s.codebook_size, splits,
                                                              reinterpret_cast<VqPartial*>(scratch));
  MC_LAUNCH_CHECK(h, "vq_simt_kernel");
  vq_merge_kernel<<<(Mq + 255) / 256, 256, 0, stream>>>(reinterpret_cast<const VqPartial*>(scratch), Mq, splits,
                                                        reinterpret_cast<long long*>(codes), margin);
  MC_LAUNCH_CHECK(h, "vq_merge_kernel");
  return MC_OK;
}

std::vector<std::string> required_tensors(const mc_spec& s) {
  std::vector<std::string> v;
  const int n = s.n_convs;
  for (int i = 0; i < n; ++i) {
    v.push_back("enc.conv" + std::to_string(i) + ".w");
    v.push_back("enc.conv" + std::to_string(i) + ".b");
    v.push_back("dec.up" + std::to_string(i) + ".w");
    v.push_back("dec.up" + std::to_string(i) + ".b");
  }
  const char* leaves[] = {"norm1", "wqkv", "bqkv", "wo", "bo", "norm2", "w1", "b1", "w2", "b2"};
  for (int st = 0; st < 2; ++st)
    for (int l = 0; l < (st == 0 ? s.enc_layers : s.dec_layers); ++l)
      for (const char* leaf : leaves)
        v.push_back(std::string(st == 0 ? "enc" : "dec") + ".layers." + std::to_string(l) + "." + leaf);
  for (const char* nm : {"enc.norm_f", "enc.proj.w", "enc.proj.b", "vq.codebook", "vq.c2", "vq.packed", "dec.in_proj.w",
                         "dec.in_proj.b", "dec.norm_f", "rope.cos", "rope.sin"})
    v.push_back(nm);
  return v;
}

// The specs the kernels are built for (the same rules as MagiCodecSpec.validate()); empty if `s` is one of them.
std::string spec_refusal(const mc_spec& s) {
  char msg[160];
  const int n = s.n_convs;
  if (n < 2 || n > MC_MAX_CONVS) return "need 2 .. " + std::to_string(MC_MAX_CONVS) + " convs";
  if (s.n_heads < 1 || s.d_model % 64 != 0 || s.d_model / s.n_heads != 64 || s.d_model % s.n_heads != 0 ||
      s.ffn_dim < 64 || s.ffn_dim % 64 != 0 || s.codebook_dim != 16 || s.codebook_size < 256 || s.codebook_size % 256 != 0 ||
      s.conv_channels[n - 1] != s.d_model || s.enc_layers < 0 || s.dec_layers < 0)
    return "need head_dim 64, d/ffn multiples of 64, codebook_dim 16, codebook_size a multiple of 256";
  if (s.window_left < 0 || s.window_left > 96 || s.window_right < 0 || s.window_right > 32)
    return "attention window (" + std::to_string(s.window_left) + ", " + std::to_string(s.window_right) +
           ") too wide: window_left <= 96, window_right <= 32";
  for (int i = 0; i < n; ++i)
    if (s.conv_strides[i] < 1 || s.conv_channels[i] < 1) return "conv strides and channels must be positive";
  const int s0 = s.conv_strides[0], c0 = s.conv_channels[0];
  if ((s0 != 4 && s0 != 8) || c0 % 8 != 0 || 256 % (c0 / 8) != 0) {
    snprintf(msg, sizeof msg, "conv0: stride %d / channels %d unsupported (stride 4 or 8, 8 * 2^k channels up to 2048)", s0, c0);
    return msg;
  }
  for (int i = 1; i < n; ++i)
    if (s.conv_strides[i] * s.conv_channels[i - 1] % 64 != 0) {
      snprintf(msg, sizeof msg, "conv %d: stride * Cin = %d * %d is not a multiple of 64", i, s.conv_strides[i], s.conv_channels[i - 1]);
      return msg;
    }
  for (int i = 1; i + 1 < n; ++i)   // transposed convs 0 .. n-2 read d and conv_channels[n-2] .. [1] as GEMM K blocks
    if (s.conv_channels[i] % 64 != 0) {
      snprintf(msg, sizeof msg, "tconv: %d input channels are not a multiple of 64", s.conv_channels[i]);
      return msg;
    }
  return std::string();
}

}  // namespace

// =============================================================== C ABI
extern "C" {

int mc_version(void) { return MC_VERSION; }

const char* mc_last_error(const mc_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int mc_create(const mc_spec* spec, int device, mc_handle** out) {
  if (!spec || !out) { g_create_error = "mc_create: null argument"; return MC_ERR_ARG; }
  *out = nullptr;
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) { g_create_error = std::string("mc_create: ") + cudaGetErrorString(e); return MC_ERR_CUDA; }
  if (prop.major != 10) {
    g_create_error = "mc_create: device is sm_" + std::to_string(prop.major * 10 + prop.minor) +
                     "; this library contains sm_100a code only (no fallback)";
    return MC_ERR_ARCH;
  }
  const std::string refusal = spec_refusal(*spec);
  if (!refusal.empty()) {
    g_create_error = "mc_create: unsupported spec: " + refusal;
    return MC_ERR_ARG;
  }
  e = cudaSetDevice(device);
  if (e != cudaSuccess) { g_create_error = std::string("mc_create: ") + cudaGetErrorString(e); return MC_ERR_CUDA; }
  mc_handle* h = new mc_handle();
  h->spec = *spec;
  h->device = device;
  h->num_sms = prop.multiProcessorCount;
  *out = h;
  return MC_OK;
}

int mc_destroy(mc_handle* h) {
  if (!h) return MC_OK;
  if (h->arena) cudaFree(h->arena);
  delete h;
  return MC_OK;
}

int mc_set_tensor(mc_handle* h, const char* name, const void* dev_ptr, int64_t numel) {
  if (!h || !name || !dev_ptr) return MC_ERR_ARG;
  Tensor t; t.p = dev_ptr; t.numel = numel;
  h->tensors[name] = t;
  h->tensor_gen++;            // captured graphs carry the old pointer: sessions re-capture (run_or_replay)
  h->finalized = false;
  return MC_OK;
}

int mc_finalize(mc_handle* h) {
  if (!h) return MC_ERR_ARG;
  for (const std::string& nm : required_tensors(h->spec))
    if (!h->find(nm)) return h->fail(MC_ERR_ARG, "mc_finalize: tensor '%s' was not registered", nm.c_str());
  h->finalized = true;
  return MC_OK;
}

#define MC_ENTER(h)                                                        \
  if (!(h)) return MC_ERR_ARG;                                             \
  if (!(h)->finalized) return (h)->fail(MC_ERR_STATE, "handle not finalized"); \
  { cudaError_t e__ = cudaSetDevice((h)->device); if (e__ != cudaSuccess) return (h)->fail(MC_ERR_CUDA, "cudaSetDevice failed"); }

int mc_encode(mc_handle* h, const float* wav, int64_t ld, int32_t B, int32_t T, int32_t keep_last_frames,
              int64_t* codes, float* margin, float* z_e, mc_stream_t stream) {
  MC_ENTER(h);
  if (!wav || !codes || B < 1 || T < 1) return h->fail(MC_ERR_ARG, "mc_encode: bad arguments (B=%d T=%d)", B, T);
  return encode_impl(h, wav, ld, B, T, keep_last_frames, codes, margin, z_e, (cudaStream_t)stream);
}

int mc_decode(mc_handle* h, const int64_t* codes, int32_t B, int32_t F, int32_t keep_last_samples, float* wav,
              mc_stream_t stream) {
  MC_ENTER(h);
  if (!codes || !wav) return h->fail(MC_ERR_ARG, "mc_decode: null pointer");
  return decode_impl(h, codes, nullptr, B, F, keep_last_samples, wav, (cudaStream_t)stream);
}

int mc_decode_latents(mc_handle* h, const float* z_q, int32_t B, int32_t F, int32_t keep_last_samples, float* wav,
                      mc_stream_t stream) {
  MC_ENTER(h);
  if (!z_q || !wav) return h->fail(MC_ERR_ARG, "mc_decode_latents: null pointer");
  return decode_impl(h, nullptr, z_q, B, F, keep_last_samples, wav, (cudaStream_t)stream);
}

int mc_vq_search(mc_handle* h, const float* z, int32_t M, int64_t* codes, float* margin, mc_stream_t stream) {
  MC_ENTER(h);
  if (!z || !codes || M < 1) return h->fail(MC_ERR_ARG, "mc_vq_search: bad arguments");
  Carver cv;
  cv.take(vq_scratch_bytes(h, M));
  MC_TRY(arena_reserve(h, cv.off, (cudaStream_t)stream));
  return launch_vq(h, z, M, 1, 1, codes, margin, h->arena, (cudaStream_t)stream);
}

int mc_codebook(mc_handle* h, float* out, mc_stream_t stream) {
  MC_ENTER(h);
  const Tensor* t = h->find("vq.codebook");
  MC_CUDA(h, cudaMemcpyAsync(out, t->p, (size_t)t->numel * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return MC_OK;
}

int mc_embed_distance(mc_handle* h, const int64_t* ids, int32_t rows, int32_t n, int64_t vocab_start, const float* ref,
                      float* dist_out, float* mean_out, mc_stream_t stream) {
  MC_ENTER(h);
  if (!ids || rows < 1 || n < 1 || (!dist_out && !mean_out)) return h->fail(MC_ERR_ARG, "mc_embed_distance: bad arguments");
  embed_distance_kernel<<<rows, POST_THREADS, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const long long*>(ids), n, (long long)vocab_start, h->ptr<float>("vq.codebook"), h->spec.codebook_size,
      ref, dist_out, mean_out);
  MC_LAUNCH_CHECK(h, "embed_distance_kernel");
  return MC_OK;
}

int mc_op_embed_distance(mc_handle* h, const float* table, int32_t K, const int64_t* ids, int32_t rows, int32_t n,
                         int64_t vocab_start, const float* ref, float* dist_out, float* mean_out, mc_stream_t stream) {
  MC_ENTER(h);
  if (!table || K < 1 || !ids || rows < 1 || n < 1 || (!dist_out && !mean_out))
    return h->fail(MC_ERR_ARG, "mc_op_embed_distance: bad arguments");
  embed_distance_kernel<<<rows, POST_THREADS, 0, (cudaStream_t)stream>>>(reinterpret_cast<const long long*>(ids), n,
                                                                         (long long)vocab_start, table, K, ref, dist_out, mean_out);
  MC_LAUNCH_CHECK(h, "embed_distance_kernel");
  return MC_OK;
}

int mc_op_emit_chunk(mc_handle* h, const float* wav, int32_t n_have, int32_t chunk, int32_t fade, int32_t has_prev,
                     float target_rms, float silence_rms_threshold, const float* fade_in, float* prev_tail, float* out,
                     mc_stream_t stream) {
  MC_ENTER(h);
  if (!wav || !fade_in || !prev_tail || !out || chunk < 1 || fade < 1 || fade > chunk || n_have < 1)
    return h->fail(MC_ERR_ARG, "mc_op_emit_chunk: bad arguments");
  emit_chunk_kernel<<<1, POST_THREADS, 0, (cudaStream_t)stream>>>(wav, n_have, chunk, fade, has_prev, target_rms,
                                                                  silence_rms_threshold, fade_in, prev_tail, out);
  MC_LAUNCH_CHECK(h, "emit_chunk_kernel");
  return MC_OK;
}

int mc_render_chunks(mc_handle* h, const float* windows, int64_t ld, int32_t n_chunks, int32_t chunk, int32_t fade,
                     int32_t last_len, float target_rms, float silence_rms_threshold, const float* fade_in, float* out,
                     mc_stream_t stream) {
  MC_ENTER(h);
  if (!windows || !fade_in || !out || n_chunks < 1 || chunk < 1 || fade < 1 || fade > chunk || last_len < 1 || last_len > chunk ||
      ld < (int64_t)chunk + fade)
    return h->fail(MC_ERR_ARG, "mc_render_chunks: need 0 < fade (%d) <= chunk (%d), 0 < last_len (%d) <= chunk, ld (%lld) >= chunk + fade",
                   fade, chunk, last_len, (long long)ld);
  const double out_n = (double)(n_chunks - 1) * chunk + last_len;
  McProfScope prof(h, 3, 0.0, out_n * 4.0 * 2.0 + (double)n_chunks * fade * 4.0, (cudaStream_t)stream);
  mc_launch(h, emit_chunks_kernel, dim3(n_chunks), dim3(POST_THREADS), 0, (cudaStream_t)stream, windows, (long long)ld, (int)n_chunks,
            (int)chunk, (int)fade, (int)last_len, target_rms, silence_rms_threshold, fade_in, out);
  MC_LAUNCH_CHECK(h, "emit_chunks_kernel");
  return MC_OK;
}

int mc_op_f32_to_pcm(mc_handle* h, const float* in, int64_t in_ld, int32_t channels, int64_t frames, int32_t format, void* out,
                     mc_stream_t stream) {
  MC_ENTER(h);
  if (!in || !out || channels < 1 || frames < 1 || in_ld < frames || (format != PCM_S16 && format != PCM_F32))
    return h->fail(MC_ERR_ARG, "mc_op_f32_to_pcm: bad arguments (format %d, channels %d, frames %lld)", format, channels, (long long)frames);
  if (reinterpret_cast<uintptr_t>(out) & (format == PCM_S16 ? 1 : 3))
    return h->fail(MC_ERR_ARG, "mc_op_f32_to_pcm: output is not naturally aligned");
  McProfScope prof(h, 3, 0.0, (double)frames * channels * (4.0 + (format == PCM_S16 ? 2.0 : 4.0)), (cudaStream_t)stream);
  f32_to_pcm_kernel<<<ew_grid(h, frames * channels, 256), 256, 0, (cudaStream_t)stream>>>(in, (long long)in_ld, channels,
                                                                                          (long long)frames, format, out);
  MC_LAUNCH_CHECK(h, "f32_to_pcm_kernel");
  return MC_OK;
}

int mc_op_pcm_to_f32(mc_handle* h, const void* pcm, int32_t format, int32_t big_endian, int32_t channels, int64_t frames,
                     int32_t mix_mono, float* out, int64_t out_ld, mc_stream_t stream) {
  MC_ENTER(h);
  if (!pcm || !out || channels < 1 || frames < 1 || format < PCM_U8 || format > PCM_ALAW || (!mix_mono && out_ld < frames))
    return h->fail(MC_ERR_ARG, "mc_op_pcm_to_f32: bad arguments (format %d, channels %d, frames %lld)", format, channels, (long long)frames);
  if ((format == PCM_F32 && (reinterpret_cast<uintptr_t>(pcm) & 3)) || (format == PCM_F64 && (reinterpret_cast<uintptr_t>(pcm) & 7)))
    return h->fail(MC_ERR_ARG, "mc_op_pcm_to_f32: float payload is not naturally aligned");
  McProfScope prof(h, 3, 0.0, (double)frames * channels * 2.0 + (double)frames * (mix_mono ? 1 : channels) * 4.0, (cudaStream_t)stream);
  pcm_to_f32_kernel<<<ew_grid(h, frames, 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const unsigned char*>(pcm), format, big_endian, channels, (long long)frames, mix_mono, out, (long long)out_ld);
  MC_LAUNCH_CHECK(h, "pcm_to_f32_kernel");
  return MC_OK;
}

int mc_op_resample(mc_handle* h, const float* in, int64_t in_ld, int32_t channels, int64_t n_in, int32_t up, int32_t down,
                   const float* taps, int32_t n_taps, int64_t pre_remove, float* out, int64_t out_ld, int64_t n_out,
                   mc_stream_t stream) {
  MC_ENTER(h);
  if (!in || !taps || !out || channels < 1 || n_in < 1 || n_out < 1 || up < 1 || down < 1 || n_taps < 1 || pre_remove < 0 ||
      in_ld < n_in || out_ld < n_out)
    return h->fail(MC_ERR_ARG, "mc_op_resample: bad arguments (up %d, down %d, taps %d)", up, down, n_taps);
  McProfScope prof(h, 3, 2.0 * channels * (double)n_out * ((double)n_taps / up), (double)channels * (n_in + n_out) * 4.0, (cudaStream_t)stream);
  resample_poly_kernel<<<ew_grid(h, (long long)channels * n_out, 256), 256, 0, (cudaStream_t)stream>>>(
      in, (long long)in_ld, channels, (long long)n_in, up, down, taps, n_taps, (long long)pre_remove, out, (long long)out_ld,
      (long long)n_out);
  MC_LAUNCH_CHECK(h, "resample_poly_kernel");
  return MC_OK;
}

/* Timeline build only (-DMC_TRACE): point the kernels' wait-time log at dev_buf (4 x uint64 per record: grid<<32|block,
 * block size, timer before / after griddepcontrol.wait); dev_buf = NULL stops logging.  Returns the records logged so far. */
int64_t mc_debug_trace(mc_handle* h, void* dev_buf, int64_t capacity_records) {
  if (!h) return MC_ERR_ARG;
#ifdef MC_TRACE
  unsigned int n = 0, zero = 0, cap = (unsigned int)capacity_records;
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(&n, g_mc_trace_n, sizeof(n));
  unsigned long long* ptr = reinterpret_cast<unsigned long long*>(dev_buf);
  cudaMemcpyToSymbol(g_mc_trace, &ptr, sizeof(ptr));
  cudaMemcpyToSymbol(g_mc_trace_cap, &cap, sizeof(cap));
  cudaMemcpyToSymbol(g_mc_trace_n, &zero, sizeof(zero));
  return (int64_t)n;
#else
  (void)dev_buf; (void)capacity_records;
  return h->fail(MC_ERR_STATE, "mc_debug_trace: the library was built without -DMC_TRACE");
#endif
}

int64_t mc_launch_count(const mc_handle* h) { return h ? h->launches : 0; }

int mc_profile_begin(mc_handle* h) {
  if (!h) return MC_ERR_ARG;
  for (auto& r : h->prof) { h->event_pool.push_back(r.a); h->event_pool.push_back(r.b); }
  h->prof.clear();
  h->profiling = true;
  return MC_OK;
}

int mc_profile_end(mc_handle* h, double* ms, double* flops, double* bytes, int64_t* launches, int32_t n_classes) {
  if (!h || !ms || !flops || !bytes || !launches) return MC_ERR_ARG;
  h->profiling = false;
  for (int c = 0; c < n_classes; ++c) { ms[c] = 0; flops[c] = 0; bytes[c] = 0; launches[c] = 0; }
  for (auto& r : h->prof) {
    cudaError_t e = cudaEventSynchronize(r.b);
    if (e != cudaSuccess) return h->fail(MC_ERR_CUDA, "mc_profile_end: %s", cudaGetErrorString(e));
    float t = 0.f;
    cudaEventElapsedTime(&t, r.a, r.b);
    if (r.cls < n_classes) { ms[r.cls] += t; flops[r.cls] += r.flops; bytes[r.cls] += r.bytes; launches[r.cls]++; }
    h->event_pool.push_back(r.a); h->event_pool.push_back(r.b);
  }
  h->prof.clear();
  return MC_OK;
}

int mc_set_option(mc_handle* h, const char* key, int32_t value) {
  if (!h || !key) return MC_ERR_ARG;
  const std::string k(key);
  if (k == "shared_stem") h->shared_stem = value != 0;
  else if (k == "exact_cut") { h->exact_cut = value != 0; h->tensor_gen++; }
  else if (k == "gemm_pair") h->gemm_pair = value != 0;
  else if (k == "fast_epilogue") h->fast_epilogue = value != 0;
  else if (k == "pdl") h->pdl = value != 0;
  else if (k == "attn_p_tmem") h->attn_p_tmem = value != 0;
  else if (k == "debug_repeat") h->debug_repeat = value;   // mc_op_* launch their kernel `value` times back to back (timing tools)
  else if (k == "l2_prefetch") { h->l2_prefetch = value != 0; h->tensor_gen++; }
  else if (k == "fuse_norm") {
    if (value < 0 || value > 3) return h->fail(MC_ERR_ARG, "mc_set_option: fuse_norm is 0 .. 3");
    h->fuse_norm = value; h->tensor_gen++;
  }
  else if (k == "small_m_split_k") {   // 0 never, 1 streaming sessions only (default), 2 every GEMM of <= 256 rows
    if (value < 0 || value > 2) return h->fail(MC_ERR_ARG, "mc_set_option: small_m_split_k is 0, 1 or 2");
    h->split_k = value;
    h->tensor_gen++;                   // sessions re-capture their graphs with the other kernels
  }
  else if (k == "max_positions") {   // rows of the re-registered rope.cos / rope.sin tables (B200Generator grows them on demand)
    if (value < 1) return h->fail(MC_ERR_ARG, "mc_set_option: max_positions must be positive");
    h->spec.max_positions = value;
  }
  else return h->fail(MC_ERR_ARG, "mc_set_option: unknown option '%s'", key);
  return MC_OK;
}

int mc_set_debug_impl(mc_handle* h, int32_t attention_impl, int32_t vq_impl) {
  if (!h) return MC_ERR_ARG;
  h->gemm_pair = (attention_impl & 4) ? 0 : 1;   // bit 2: force the single-CTA GEMM (A/B measurements)
  attention_impl &= 1;
  h->attn_impl = attention_impl;
  h->vq_impl = vq_impl;
  return MC_OK;
}

int mc_op_gemm(mc_handle* h, const void* A, int64_t a_rows, int32_t a_k_wrap, const void* W, const float* bias,
               int32_t M, int32_t N, int32_t K, int32_t act, int32_t out_mode, void* out, int64_t ldo,
               int32_t grp_in, int32_t grp_valid, int64_t grp_stride, int64_t grp_off, int32_t rope_cols,
               int32_t rope_period, int32_t block_n, mc_stream_t stream) {
  MC_ENTER(h);
  GemmCall g{};
  g.A = reinterpret_cast<const bf16*>(A); g.a_rows = a_rows; g.a_k_wrap = a_k_wrap;
  g.W = reinterpret_cast<const bf16*>(W); g.bias = bias; g.M = M; g.N = N; g.K = K; g.act = act; g.out_mode = out_mode;
  g.out = out; g.ldo = ldo;
  g.grp_in = grp_in > 0 ? grp_in : INT_MAX; g.grp_valid = grp_in > 0 ? grp_valid : INT_MAX;
  g.grp_stride = grp_stride; g.grp_off = grp_off;
  g.rope_cols = rope_cols; g.rope_period = rope_period; g.block_n = block_n;
  for (int r = 1; r < h->debug_repeat; ++r) MC_TRY(launch_gemm(h, g, (cudaStream_t)stream));   // back-to-back chain (timing)
  return launch_gemm(h, g, (cudaStream_t)stream);
}

/* Plain GEMM with the fused-RMSNorm roles (GemmParams): consumer (row_stats [M, row_stats_n] -> y = acc * rs(row) + bias)
 * and / or producer (fp32 output modes: also xb_out = bf16(x_new * xb_gamma) [M, N] and stat_out [M, N/64]). */
int mc_op_gemm_fused(mc_handle* h, const void* A, const void* W, const float* bias, int32_t M, int32_t N, int32_t K, int32_t act,
                     int32_t out_mode, void* out, const float* row_stats, int32_t row_stats_n, void* xb_out, const float* xb_gamma,
                     float* stat_out, int32_t rope_cols, int32_t rope_period, int32_t block_n, mc_stream_t stream) {
  MC_ENTER(h);
  GemmCall g{};
  g.A = reinterpret_cast<const bf16*>(A); g.a_rows = M; g.a_k_wrap = K;
  g.W = reinterpret_cast<const bf16*>(W); g.bias = bias; g.M = M; g.N = N; g.K = K; g.act = act; g.out_mode = out_mode;
  g.out = out; g.ldo = N;
  g.rope_cols = rope_cols; g.rope_period = rope_period; g.block_n = block_n;
  g.row_stats = row_stats; g.row_stats_n = row_stats_n;
  g.xb_out = reinterpret_cast<bf16*>(xb_out); g.xb_gamma = xb_gamma; g.stat_out = stat_out;
  for (int r = 1; r < h->debug_repeat; ++r) MC_TRY(launch_gemm(h, g, (cudaStream_t)stream));   // back-to-back chain (timing)
  return launch_gemm(h, g, (cudaStream_t)stream);
}

int mc_op_rowstats(mc_handle* h, const float* x, const float* gamma, void* xb_out, float* stat_out, int32_t M, int32_t d,
                   mc_stream_t stream) {
  MC_ENTER(h);
  if (!x || !gamma || !xb_out || !stat_out || M < 1 || d % 64 != 0) return h->fail(MC_ERR_ARG, "mc_op_rowstats: bad arguments");
  for (int r = 1; r < h->debug_repeat; ++r) MC_TRY(launch_rowstats(h, x, gamma, reinterpret_cast<bf16*>(xb_out), stat_out, M, d, (cudaStream_t)stream));
  return launch_rowstats(h, x, gamma, reinterpret_cast<bf16*>(xb_out), stat_out, M, d, (cudaStream_t)stream);
}

int mc_op_rmsnorm(mc_handle* h, const float* x, const float* gamma, void* out_bf16, int32_t M, int32_t d,
                  mc_stream_t stream) {
  MC_ENTER(h);
  for (int r = 1; r < h->debug_repeat; ++r) MC_TRY(launch_rmsnorm(h, x, gamma, reinterpret_cast<bf16*>(out_bf16), M, d, INT_MAX, 0, 0, (cudaStream_t)stream));
  return launch_rmsnorm(h, x, gamma, reinterpret_cast<bf16*>(out_bf16), M, d, INT_MAX, 0, 0, (cudaStream_t)stream);
}

int mc_op_attention(mc_handle* h, const void* qkv, void* out, int32_t B, int32_t F, int32_t out_rows, int32_t phase,
                    int32_t impl, mc_stream_t stream) {
  MC_ENTER(h);
  for (int r = 1; r < h->debug_repeat; ++r)
    MC_TRY(launch_attention(h, reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(out), B, F, out_rows, phase, impl,
                            (cudaStream_t)stream));
  return launch_attention(h, reinterpret_cast<const bf16*>(qkv), reinterpret_cast<bf16*>(out), B, F, out_rows, phase, impl,
                          (cudaStream_t)stream);
}

}  // extern "C"

// =====================================================================================
// Streaming sessions (SURVEY §8b): the rolling 2.0 s context of AudioTokenizer.tokenize_audio /
// detokenize_audio (audio_tokenizer.py:72-74,111-113) kept resident in HBM.  Each push uploads only
// the new chunk, rebuilds the context in a ping-pong buffer, runs the batched encode/decode over the
// channels and returns the kept frames/samples through pinned staging.  The whole sequence for a
// given (context length, chunk length, keep) is captured once into a CUDA graph and replayed: the
// steady state of the full-duplex loop is ONE graph launch per call.
// =====================================================================================
struct mc_stream {
  mc_handle* h = nullptr;
  int C = 1;
  int ctx_samples = 32000, ctx_frames = 100;
  int cap_samples = 0, cap_frames = 0;
  float* audio[2] = {nullptr, nullptr};
  int64_t* codes_ctx[2] = {nullptr, nullptr};
  int audio_len = 0, code_len = 0, acur = 0, ccur = 0;
  int32_t* pin_table = nullptr; // {0, current context buffer}: read in place by the roll kernel
  float* pin_audio = nullptr;   // [C, cap_samples]
  int64_t* pin_codes = nullptr; // [C, cap_frames]
  float* pin_wav = nullptr;     // [C, cap_samples]
  int64_t* dev_codes_out = nullptr;
  float* dev_wav_out = nullptr;
  struct GraphEntry { cudaGraphExec_t exec = nullptr; int uses = 0; size_t arena_gen = 0; };
  std::map<std::tuple<int, int, int, int, int>, GraphEntry> graphs;  // (kind, len_before, n, keep, parity)
  bool use_graphs = true;
  // work runs on the session's own stream (the caller's may be the legacy default stream, which cannot be
  // captured); each push first orders it after everything already queued on the caller's stream
  cudaStream_t own = nullptr;
  cudaEvent_t order_ev = nullptr;
  std::string err;
  // post-decode emit chain (mc_stream_set_emit / mc_stream_push_codes_emit)
  int emit_chunk = 0, emit_fade = 0, emit_has_prev = 0;
  float emit_target_rms = 0.f, emit_silence_thr = 0.f;
  float* emit_fade_in = nullptr;   // device [fade]
  float* emit_prev_tail = nullptr; // device [fade]
  float* emit_out = nullptr;       // device [2*chunk + fade]
  float* pin_emit = nullptr;       // pinned  [2*chunk + fade]
};

namespace {

// everything a captured graph bakes in besides its key: the workspace arena and the registered tensors
size_t handle_generation(const mc_handle* h) {
  return reinterpret_cast<size_t>(h->arena) ^ h->arena_cap ^ (static_cast<size_t>(h->tensor_gen) << 48);
}

void stream_drop_graphs(mc_stream* s) {
  for (auto& kv : s->graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  s->graphs.clear();
}

// Runs `body` directly the first time a key is seen (that run sizes the workspace and fills the TMA
// descriptor cache), captures it into a graph the second time, and replays the graph afterwards.
template <typename Sess, typename Key, typename Body>
int run_or_replay_impl(Sess* s, Key key, cudaStream_t stream, Body body);

// Everything a session launches (directly or while capturing) is "in session": few-rows GEMMs take the split-K kernels.
template <typename Sess, typename Key, typename Body>
int run_or_replay(Sess* s, Key key, cudaStream_t stream, Body body) {
  s->h->in_session = true;
  const int rc = run_or_replay_impl(s, key, stream, body);
  s->h->in_session = false;
  return rc;
}

template <typename Sess, typename Key, typename Body>
int run_or_replay_impl(Sess* s, Key key, cudaStream_t stream, Body body) {
  mc_handle* h = s->h;
  if (!s->use_graphs || h->profiling) return body();
  auto& e = s->graphs[key];
  const size_t gen = handle_generation(h);
  if (e.exec && e.arena_gen != gen) {
    cudaGraphExecDestroy(e.exec);
    e.exec = nullptr;
    e.uses = 0;
  }
  if (e.exec) {
    MC_CUDA(h, cudaGraphLaunch(e.exec, stream));
    h->launches += 1;
    return MC_OK;
  }
  if (e.uses++ == 0) return body();
  MC_CUDA(h, cudaStreamBeginCapture(stream, cudaStreamCaptureModeRelaxed));
  const int64_t launches_before = h->launches;
  const int rc = body();
  cudaGraph_t graph = nullptr;
  cudaError_t ce = cudaStreamEndCapture(stream, &graph);
  h->launches = launches_before;
  if (rc != MC_OK || ce != cudaSuccess || graph == nullptr) {
    if (graph) cudaGraphDestroy(graph);
    (void)cudaGetLastError();
    s->use_graphs = false;  // fall back to direct launches for this session
    return body();
  }
  ce = cudaGraphInstantiate(&e.exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ce != cudaSuccess) {
    e.exec = nullptr;
    s->use_graphs = false;
    return body();
  }
  e.arena_gen = handle_generation(h);
  MC_CUDA(h, cudaGraphLaunch(e.exec, stream));
  h->launches += 1;
  return MC_OK;
}

}  // namespace

extern "C" {

int mc_stream_create(mc_handle* h, int32_t channels, int32_t context_samples, int32_t max_chunk_samples, mc_stream** out) {
  MC_ENTER(h);
  if (!out || channels < 1 || context_samples < 1) return h->fail(MC_ERR_ARG, "mc_stream_create: bad arguments");
  int hop = 1;
  for (int i = 0; i < h->spec.n_convs; ++i) hop *= h->spec.conv_strides[i];
  mc_stream* s = new mc_stream();
  s->h = h; s->C = channels;
  s->ctx_samples = context_samples;
  s->ctx_frames = context_samples / hop;
  s->cap_samples = std::max(context_samples, max_chunk_samples);
  s->cap_frames = (s->cap_samples + hop - 1) / hop;
  if (s->cap_frames > h->spec.max_positions) { delete s; return h->fail(MC_ERR_ARG, "mc_stream_create: context exceeds RoPE table"); }
  const size_t ab = (size_t)channels * s->cap_samples * 4, cb = (size_t)channels * s->cap_frames * 8;
  cudaError_t e = cudaSuccess;
  for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
    e = cudaMalloc(&s->audio[i], ab);
    if (e == cudaSuccess) e = cudaMalloc(&s->codes_ctx[i], cb);
  }
  if (e == cudaSuccess) e = cudaMalloc(&s->dev_codes_out, cb);
  if (e == cudaSuccess) e = cudaMalloc(&s->dev_wav_out, ab);
  if (e == cudaSuccess) e = cudaMallocHost(&s->pin_table, 16);
  if (e == cudaSuccess) e = cudaMallocHost(&s->pin_audio, ab);
  if (e == cudaSuccess) e = cudaMallocHost(&s->pin_codes, cb);
  if (e == cudaSuccess) e = cudaMallocHost(&s->pin_wav, ab);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->own, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->order_ev, cudaEventDisableTiming);
  if (e != cudaSuccess) { mc_stream_destroy(s); return h->fail(MC_ERR_NOMEM, "mc_stream_create: %s", cudaGetErrorString(e)); }
  *out = s;
  return MC_OK;
}

int mc_stream_destroy(mc_stream* s) {
  if (!s) return MC_OK;
  stream_drop_graphs(s);
  for (int i = 0; i < 2; ++i) { if (s->audio[i]) cudaFree(s->audio[i]); if (s->codes_ctx[i]) cudaFree(s->codes_ctx[i]); }
  if (s->dev_codes_out) cudaFree(s->dev_codes_out);
  if (s->dev_wav_out) cudaFree(s->dev_wav_out);
  if (s->pin_table) cudaFreeHost(s->pin_table);
  if (s->pin_audio) cudaFreeHost(s->pin_audio);
  if (s->pin_codes) cudaFreeHost(s->pin_codes);
  if (s->pin_wav) cudaFreeHost(s->pin_wav);
  if (s->emit_fade_in) cudaFree(s->emit_fade_in);
  if (s->emit_prev_tail) cudaFree(s->emit_prev_tail);
  if (s->emit_out) cudaFree(s->emit_out);
  if (s->pin_emit) cudaFreeHost(s->pin_emit);
  if (s->order_ev) cudaEventDestroy(s->order_ev);
  if (s->own) cudaStreamDestroy(s->own);
  delete s;
  return MC_OK;
}

int mc_stream_reset(mc_stream* s) {
  if (!s) return MC_ERR_ARG;
  s->audio_len = 0; s->code_len = 0;
  s->emit_has_prev = 0;
  return MC_OK;
}

int mc_stream_reset_part(mc_stream* s, int32_t audio, int32_t codes) {
  if (!s) return MC_ERR_ARG;
  if (audio) s->audio_len = 0;
  if (codes) s->code_len = 0;
  return MC_OK;
}

/* Context upload without compute: the session's audio (codes) context becomes the last min(n, context) samples
 * (frames) of the HOST array [C, n].  Used to re-seed a session after a one-shot call changed the host-side context
 * (AudioTokenizer keeps both in step); synchronous. */
int mc_stream_load_audio(mc_stream* s, const float* audio, int32_t n) {
  if (!s) return MC_ERR_ARG;
  mc_handle* h = s->h;
  MC_ENTER(h);
  if (n < 0 || (n > 0 && !audio)) return h->fail(MC_ERR_ARG, "mc_stream_load_audio: bad arguments");
  const int keep = std::min(n, s->ctx_samples);
  MC_CUDA(h, cudaStreamSynchronize(s->own));
  if (keep > 0)
    MC_CUDA(h, cudaMemcpy2D(s->audio[s->acur], (size_t)s->cap_samples * 4, audio + (n - keep), (size_t)n * 4, (size_t)keep * 4,
                            s->C, cudaMemcpyHostToDevice));
  s->audio_len = keep;
  return MC_OK;
}

int mc_stream_load_codes(mc_stream* s, const int64_t* codes, int32_t n) {
  if (!s) return MC_ERR_ARG;
  mc_handle* h = s->h;
  MC_ENTER(h);
  if (n < 0 || (n > 0 && !codes)) return h->fail(MC_ERR_ARG, "mc_stream_load_codes: bad arguments");
  const int keep = std::min(n, s->ctx_frames);
  MC_CUDA(h, cudaStreamSynchronize(s->own));
  if (keep > 0)
    MC_CUDA(h, cudaMemcpy2D(s->codes_ctx[s->ccur], (size_t)s->cap_frames * 8, codes + (n - keep), (size_t)n * 8, (size_t)keep * 8,
                            s->C, cudaMemcpyHostToDevice));
  s->code_len = keep;
  return MC_OK;
}

/* chunk: HOST fp32 [C, n] (row stride n).  The context becomes the last max(n, context) samples of
 * (context ++ chunk) — audio_tokenizer.py:72-74.  codes_out: HOST int64 [C, keep_frames] = the last
 * keep_frames frames of the window (0 = all); *frames_out = frames written per channel.  Synchronises
 * the stream before returning (the caller needs the codes). */
int mc_stream_push_audio(mc_stream* s, const float* chunk, int32_t n, int32_t keep_frames, int64_t* codes_out,
                         int32_t* frames_out, mc_stream_t stream_) {
  if (!s) return MC_ERR_ARG;
  mc_handle* h = s->h;
  MC_ENTER(h);
  cudaStream_t caller = (cudaStream_t)stream_;
  MC_CUDA(h, cudaEventRecord(s->order_ev, caller));
  MC_CUDA(h, cudaStreamWaitEvent(s->own, s->order_ev, 0));
  cudaStream_t stream = s->own;
  if (!chunk || !codes_out || n < 1) return h->fail(MC_ERR_ARG, "mc_stream_push_audio: bad arguments");
  if (n > s->cap_samples) return h->fail(MC_ERR_ARG, "mc_stream_push_audio: chunk of %d samples exceeds the session capacity %d", n, s->cap_samples);
  int hop = 1;
  for (int i = 0; i < h->spec.n_convs; ++i) hop *= h->spec.conv_strides[i];
  const int C = s->C, cap = s->cap_samples;
  const int new_len = std::min(s->audio_len + n, std::max(n, s->ctx_samples));
  const int keep_old = new_len - n;
  const int F = (new_len + hop - 1) / hop;
  const int keep = (keep_frames <= 0 || keep_frames > F) ? F : keep_frames;
  for (int c = 0; c < C; ++c) memcpy(s->pin_audio + (size_t)c * cap, chunk + (size_t)c * n, (size_t)n * 4);
  const int src = s->acur, dst = s->acur ^ 1;
  const int old_len = s->audio_len;
  // One kernel rolls the context (kept tail ++ the new chunk, read in place from pinned host memory) and the last
  // kernel of the pass writes the codes straight into pinned host memory: no copy nodes on the latency path.
  s->pin_table[0] = 0; s->pin_table[1] = src;
  auto body = [&]() -> int {
    pool_roll_kernel<float><<<dim3((new_len + 255) / 256, C), 256, 0, stream>>>(s->pin_table, C, cap, old_len, keep_old, n, s->audio[0],
                                                                               s->audio[1], s->pin_audio, nullptr, 0);
    MC_LAUNCH_CHECK(h, "pool_roll_kernel");
    MC_TRY(encode_impl(h, s->audio[dst], cap, C, new_len, keep, s->pin_codes, nullptr, nullptr, stream));
    return MC_OK;
  };
  MC_TRY(run_or_replay(s, std::make_tuple(0, old_len, n, keep, src), stream, body));
  MC_CUDA(h, cudaStreamSynchronize(stream));
  memcpy(codes_out, s->pin_codes, (size_t)C * keep * 8);
  if (frames_out) *frames_out = keep;
  s->acur = dst;
  s->audio_len = new_len;
  return MC_OK;
}

/* codes: HOST int64 [C, n] appended to the code context (last max(n, context_frames) frames kept,
 * audio_tokenizer.py:111-113); wav_out: HOST fp32 [C, keep_samples] = the last keep_samples samples of
 * the decoded window (0 = all); *samples_out = samples written per channel.
 * emit = true (mc_stream_push_codes_emit): keep = chunk + fade samples, followed IN THE SAME GRAPH by
 * emit_chunk_kernel; wav_out then receives the kernel's [2*chunk + fade] output block. */
static int stream_push_codes_impl(mc_stream* s, const int64_t* codes, int32_t n, int32_t keep_samples, bool emit,
                                  float* wav_out, int32_t* samples_out, mc_stream_t stream_) {
  if (!s) return MC_ERR_ARG;
  mc_handle* h = s->h;
  MC_ENTER(h);
  cudaStream_t caller = (cudaStream_t)stream_;
  MC_CUDA(h, cudaEventRecord(s->order_ev, caller));
  MC_CUDA(h, cudaStreamWaitEvent(s->own, s->order_ev, 0));
  cudaStream_t stream = s->own;
  if (!codes || !wav_out || n < 1) return h->fail(MC_ERR_ARG, "mc_stream_push_codes: bad arguments");
  if (n > s->cap_frames) return h->fail(MC_ERR_ARG, "mc_stream_push_codes: %d frames exceed the session capacity %d", n, s->cap_frames);
  int hop = 1;
  for (int i = 0; i < h->spec.n_convs; ++i) hop *= h->spec.conv_strides[i];
  const int C = s->C, cap = s->cap_frames;
  const int new_len = std::min(s->code_len + n, std::max(n, s->ctx_frames));
  const int keep_old = new_len - n;
  const int total = new_len * hop;
  int keep = (keep_samples <= 0 || keep_samples > total) ? total : keep_samples;
  const int has_prev = s->emit_has_prev;
  if (emit) {
    if (C != 1) return h->fail(MC_ERR_ARG, "mc_stream_push_codes_emit: the emit chain is mono (pad_or_trim rejects [C,T])");
    if (s->emit_chunk <= 0) return h->fail(MC_ERR_STATE, "mc_stream_push_codes_emit: call mc_stream_set_emit first");
    if (n * hop != s->emit_chunk)
      return h->fail(MC_ERR_ARG, "mc_stream_push_codes_emit: %d codes decode to %d samples, chunk is %d", n, n * hop, s->emit_chunk);
    keep = std::min(total, s->emit_chunk + s->emit_fade);
    // realtime_agent_v2.py:566-568 asserts the joined length; the same conditions fail here, before any work
    if (has_prev && keep != s->emit_chunk + s->emit_fade)
      return h->fail(MC_ERR_STATE, "mc_stream_push_codes_emit: only %d decoded samples for chunk %d + fade %d", keep, s->emit_chunk, s->emit_fade);
    if (!has_prev && keep != s->emit_chunk)
      return h->fail(MC_ERR_STATE, "mc_stream_push_codes_emit: the first emitted chunk needs an empty code context (reset first)");
  }
  for (int c = 0; c < C; ++c) memcpy(s->pin_codes + (size_t)c * cap, codes + (size_t)c * n, (size_t)n * 8);
  const int src = s->ccur, dst = s->ccur ^ 1;
  const int old_len = s->code_len;
  const int emit_floats = 2 * s->emit_chunk + s->emit_fade;
  // decode_impl wants dense [C, new_len] codes: the context buffers use row stride `cap`, so gather rows densely
  s->pin_table[0] = 0; s->pin_table[1] = src;
  auto body = [&]() -> int {
    // one kernel: context roll (codes read in place from pinned host memory) + the dense [C, new_len] batch the decoder reads
    pool_roll_kernel<long long><<<dim3((new_len + 255) / 256, C), 256, 0, stream>>>(
        s->pin_table, C, cap, old_len, keep_old, n, reinterpret_cast<long long*>(s->codes_ctx[0]), reinterpret_cast<long long*>(s->codes_ctx[1]),
        reinterpret_cast<const long long*>(s->pin_codes), reinterpret_cast<long long*>(s->dev_codes_out), new_len);
    MC_LAUNCH_CHECK(h, "pool_roll_kernel");
    if (emit) {
      MC_TRY(decode_impl(h, s->dev_codes_out, nullptr, C, new_len, keep, s->dev_wav_out, stream));
      mc_launch(h, emit_chunk_kernel, dim3(1), dim3(POST_THREADS), 0, stream, (const float*)s->dev_wav_out, keep, s->emit_chunk,
                s->emit_fade, has_prev, s->emit_target_rms, s->emit_silence_thr, (const float*)s->emit_fade_in, s->emit_prev_tail,
                s->pin_emit);                                  // the emitted block lands in pinned host memory directly
      MC_LAUNCH_CHECK(h, "emit_chunk_kernel");
    } else {
      MC_TRY(decode_impl(h, s->dev_codes_out, nullptr, C, new_len, keep, s->pin_wav, stream));   // last kernel stores to pinned host memory
    }
    return MC_OK;
  };
  MC_TRY(run_or_replay(s, std::make_tuple(emit ? 2 + has_prev : 1, old_len, n, keep, src), stream, body));
  MC_CUDA(h, cudaStreamSynchronize(stream));
  if (emit) {
    memcpy(wav_out, s->pin_emit, (size_t)emit_floats * 4);
    if (samples_out) *samples_out = has_prev;
    s->emit_has_prev = 1;
  } else {
    memcpy(wav_out, s->pin_wav, (size_t)C * keep * 4);
    if (samples_out) *samples_out = keep;
  }
  s->ccur = dst;
  s->code_len = new_len;
  return MC_OK;
}

int mc_stream_push_codes(mc_stream* s, const int64_t* codes, int32_t n, int32_t keep_samples, float* wav_out,
                         int32_t* samples_out, mc_stream_t stream_) {
  return stream_push_codes_impl(s, codes, n, keep_samples, false, wav_out, samples_out, stream_);
}

int mc_stream_set_emit(mc_stream* s, int32_t chunk_samples, int32_t fade_samples, float target_rms,
                       float silence_rms_threshold, const float* fade_in) {
  if (!s) return MC_ERR_ARG;
  mc_handle* h = s->h;
  MC_ENTER(h);
  if (chunk_samples < 1 || fade_samples < 1 || fade_samples > chunk_samples || !fade_in)
    return h->fail(MC_ERR_ARG, "mc_stream_set_emit: need 0 < fade (%d) <= chunk (%d) and a ramp", fade_samples, chunk_samples);
  if (chunk_samples + fade_samples > s->cap_samples)
    return h->fail(MC_ERR_ARG, "mc_stream_set_emit: chunk + fade exceeds the session capacity %d", s->cap_samples);
  MC_CUDA(h, cudaStreamSynchronize(s->own));
  stream_drop_graphs(s);   // the captured kernels carry the old parameters
  if (s->emit_fade_in) cudaFree(s->emit_fade_in);
  if (s->emit_prev_tail) cudaFree(s->emit_prev_tail);
  if (s->emit_out) cudaFree(s->emit_out);
  if (s->pin_emit) cudaFreeHost(s->pin_emit);
  s->emit_fade_in = s->emit_prev_tail = s->emit_out = s->pin_emit = nullptr;
  const size_t fb = (size_t)std::max(1, fade_samples) * 4, ob = (size_t)(2 * chunk_samples + fade_samples) * 4;
  MC_CUDA(h, cudaMalloc(&s->emit_fade_in, fb));
  MC_CUDA(h, cudaMalloc(&s->emit_prev_tail, fb));
  MC_CUDA(h, cudaMalloc(&s->emit_out, ob));
  MC_CUDA(h, cudaMallocHost(&s->pin_emit, ob));
  if (fade_samples > 0) MC_CUDA(h, cudaMemcpy(s->emit_fade_in, fade_in, (size_t)fade_samples * 4, cudaMemcpyHostToDevice));
  MC_CUDA(h, cudaMemset(s->emit_prev_tail, 0, fb));
  s->emit_chunk = chunk_samples; s->emit_fade = fade_samples;
  s->emit_target_rms = target_rms; s->emit_silence_thr = silence_rms_threshold;
  s->emit_has_prev = 0;
  return MC_OK;
}

int mc_stream_push_codes_emit(mc_stream* s, const int64_t* codes, int32_t n, float* out, int32_t* had_prev,
                              mc_stream_t stream_) {
  return stream_push_codes_impl(s, codes, n, 0, true, out, had_prev, stream_);
}

int mc_stream_set_graphs(mc_stream* s, int32_t enabled) {
  if (!s) return MC_ERR_ARG;
  s->use_graphs = enabled != 0;
  if (!enabled) stream_drop_graphs(s);
  return MC_OK;
}

}  // extern "C"

// =====================================================================================
// Session pool: S independent rolling contexts, batched per call (SURVEY §8 f2).  tts_server.py:59 tokenizes every
// 0.1 s of every active TTS stream and realtime_agent_resources.py:41-49 runs two agents on one model: each such
// session alone is a batch-1 pass that streams all weights for 100 rows.  Sessions whose contexts have the same
// length are pushed together as ONE B = n*C launch (the Python SessionBatcher groups them), so n sessions cost about
// one.  Semantics per session are exactly mc_stream_push_audio / mc_stream_push_codes.
// =====================================================================================
struct mc_pool {
  mc_handle* h = nullptr;
  int C = 1, max_sessions = 0;
  int ctx_samples = 0, ctx_frames = 0, cap_samples = 0, cap_frames = 0;
  float* audio[2] = {nullptr, nullptr};        // [max_sessions][C][cap_samples]
  int64_t* codes[2] = {nullptr, nullptr};      // [max_sessions][C][cap_frames]
  std::vector<int> audio_len, code_len, acur, ccur;
  float *pin_chunk = nullptr, *dev_chunk = nullptr, *batch_audio = nullptr;          // [max_sessions*C][cap_samples]
  int64_t *pin_codes_in = nullptr, *dev_codes_in = nullptr, *batch_codes = nullptr;  // [max_sessions*C][cap_frames]
  int32_t *pin_table = nullptr, *dev_table = nullptr;                                // [max_sessions][2], ragged [max_sessions][4]
  int64_t *dev_codes_out = nullptr, *pin_codes_out = nullptr;
  float *dev_wav_out = nullptr, *pin_wav_out = nullptr;
  struct GraphEntry { cudaGraphExec_t exec = nullptr; int uses = 0; size_t arena_gen = 0; };
  // uniform calls: (kind 0-3, len_before, n_new, keep, batch items, 0); ragged calls: (kind 4-6, T_max or F_max, n_new,
  // cut, batch items, keep) -- the per-item lengths live in the table the graph uploads
  std::map<std::tuple<int, int, int, int, int, int>, GraphEntry> graphs;
  bool use_graphs = true;
  cudaStream_t own = nullptr;
  cudaEvent_t order_ev = nullptr;
  // post-decode emit chain shared by every slot (mc_pool_set_emit / mc_pool_push_codes_emit)
  int emit_chunk = 0, emit_fade = 0;
  float emit_target_rms = 0.f, emit_silence_thr = 0.f;
  std::vector<int> emit_has_prev;  // per slot
  float* emit_fade_in = nullptr;   // device [fade]
  float* emit_prev_tails = nullptr;// device [max_sessions][fade]
  float* pin_emit = nullptr;       // pinned [max_sessions][2*chunk + fade]
  // live-stream ingest (mc_pool_set_resampler / mc_pool_push_pcm): one polyphase plan per client rate, and the clients'
  // raw chunks staged in pinned memory, read in place by pool_ingest_kernel
  struct Resampler { int sr = 0, up = 1, down = 1, n_taps = 0; long long pre_remove = 0; float* taps = nullptr; };
  std::vector<Resampler> resamplers;
  unsigned char* pin_pcm = nullptr;
  size_t pin_pcm_bytes = 0;
  int pcm_max_in = 0, pcm_max_channels = 0;   // mc_pool_reserve_pcm's bounds (0: the staging grows when a call needs it)
  PoolIngestItem* pin_items = nullptr;         // pinned [max_sessions]
};

namespace {
void pool_drop_graphs(mc_pool* p) {
  for (auto& kv : p->graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  p->graphs.clear();
}

void pool_free_emit(mc_pool* p) {
  if (p->emit_fade_in) cudaFree(p->emit_fade_in);
  if (p->emit_prev_tails) cudaFree(p->emit_prev_tails);
  if (p->pin_emit) cudaFreeHost(p->pin_emit);
  p->emit_fade_in = p->emit_prev_tails = p->pin_emit = nullptr;
  p->emit_chunk = p->emit_fade = 0;
}

// same_len = false (ragged calls): any context lengths; *common_len = -1 when they differ.
int pool_check_slots(mc_pool* p, const int32_t* slots, int n, const std::vector<int>& lens, int* common_len, const char* what,
                     bool same_len = true) {
  mc_handle* h = p->h;
  if (!slots || n < 1 || n > p->max_sessions) return h->fail(MC_ERR_ARG, "%s: need 1..%d sessions, got %d", what, p->max_sessions, n);
  for (int j = 0; j < n; ++j) {
    if (slots[j] < 0 || slots[j] >= p->max_sessions) return h->fail(MC_ERR_ARG, "%s: slot %d out of range", what, slots[j]);
    for (int k = 0; k < j; ++k)
      if (slots[k] == slots[j]) return h->fail(MC_ERR_ARG, "%s: slot %d listed twice", what, slots[j]);
    if (same_len && lens[slots[j]] != lens[slots[0]])
      return h->fail(MC_ERR_ARG, "%s: sessions %d and %d hold contexts of different length (%d vs %d); batch them separately", what,
                     slots[0], slots[j], lens[slots[0]], lens[slots[j]]);
  }
  *common_len = lens[slots[0]];
  for (int j = 1; j < n; ++j)
    if (lens[slots[j]] != lens[slots[0]]) *common_len = -1;
  return MC_OK;
}

// Ragged calls: the pinned table of pool_roll_ragged_kernel, {slot, context buffer, old_len, new_len} per item, for
// contexts that keep the last max(len, ctx) values; returns the longest new context.
int pool_fill_ragged_table(mc_pool* p, const int32_t* slots, int n, int len, int ctx, const std::vector<int>& lens,
                           const std::vector<int>& cur) {
  int longest = 0;
  for (int j = 0; j < n; ++j) {
    const int s = slots[j], new_len = std::min(lens[s] + len, std::max(len, ctx));
    int32_t* t = p->pin_table + 4 * j;
    t[0] = s; t[1] = cur[s]; t[2] = lens[s]; t[3] = new_len;
    longest = std::max(longest, new_len);
  }
  return longest;
}

// Rows of a ragged batch's last transformer layers: rounded up to 16 to bound the number of graphs (the cut is exact at
// any depth), never more than the window.
int ragged_cut(int rows, int F) { return std::min(F, (rows + 15) / 16 * 16); }

// Decoder rows of a ragged decode whose items keep keep_j = min(keep, F_j * hop) samples each (the earliest kept sample
// over the batch, plus the frames the transposed convs look back: tconv_margin_frames), and the `keep` decode_impl takes
// for that cut.
void ragged_decode_cut(const mc_pool* p, int n, int F_max, int hop, int keep, int* rows, int* dec_keep) {
  int need = 0;
  for (int j = 0; j < n; ++j) {
    const int total_j = p->pin_table[4 * j + 3] * hop;
    need = std::max(need, (F_max * hop - total_j) + std::min(keep, total_j));
  }
  const int margin = tconv_margin_frames(p->h->spec);
  *rows = ragged_cut((need + hop - 1) / hop + margin, F_max);
  *dec_keep = *rows >= F_max ? F_max * hop : (*rows - margin) * hop;
}

int pool_hop(const mc_pool* p) {
  int hop = 1;
  for (int i = 0; i < p->h->spec.n_convs; ++i) hop *= p->h->spec.conv_strides[i];
  return hop;
}

// What mc_pool_push_audio and mc_pool_push_pcm share once the checks have passed and the new chunks are staged on the
// host: `stage(stream)` enqueues what fills dev_chunk ([n*C][cap], len samples per row); the context roll, the encode
// and the codes' way back follow in the same graph.  kind: the first element of the graph key.
template <typename Stage>
int pool_encode_uniform(mc_pool* p, const int32_t* slots, int n, int old_len, int len, int keep_frames, int64_t* codes_out,
                        int32_t* frames_out, mc_stream_t stream_, int kind, Stage stage) {
  mc_handle* h = p->h;
  MC_CUDA(h, cudaEventRecord(p->order_ev, (cudaStream_t)stream_));
  MC_CUDA(h, cudaStreamWaitEvent(p->own, p->order_ev, 0));
  cudaStream_t stream = p->own;
  const int hop = pool_hop(p);
  const int C = p->C, cap = p->cap_samples, rows = n * C;
  const int new_len = std::min(old_len + len, std::max(len, p->ctx_samples));
  const int keep_old = new_len - len;
  const int F = (new_len + hop - 1) / hop;
  const int keep = (keep_frames <= 0 || keep_frames > F) ? F : keep_frames;
  for (int j = 0; j < n; ++j) { p->pin_table[2 * j] = slots[j]; p->pin_table[2 * j + 1] = p->acur[slots[j]]; }
  auto body = [&]() -> int {
    MC_CUDA(h, cudaMemcpyAsync(p->dev_table, p->pin_table, (size_t)n * 8, cudaMemcpyHostToDevice, stream));
    MC_TRY(stage(stream));
    pool_roll_kernel<float><<<dim3((new_len + 255) / 256, rows), 256, 0, stream>>>(p->dev_table, C, cap, old_len, keep_old, len, p->audio[0],
                                                                                  p->audio[1], p->dev_chunk, p->batch_audio, cap);
    MC_LAUNCH_CHECK(h, "pool_roll_kernel");
    MC_TRY(encode_impl(h, p->batch_audio, cap, rows, new_len, keep, p->dev_codes_out, nullptr, nullptr, stream));
    MC_CUDA(h, cudaMemcpyAsync(p->pin_codes_out, p->dev_codes_out, (size_t)rows * keep * 8, cudaMemcpyDeviceToHost, stream));
    return MC_OK;
  };
  MC_TRY(run_or_replay(p, std::make_tuple(kind, old_len, len, keep, n, 0), stream, body));
  MC_CUDA(h, cudaStreamSynchronize(stream));
  memcpy(codes_out, p->pin_codes_out, (size_t)rows * keep * 8);
  if (frames_out) *frames_out = keep;
  for (int j = 0; j < n; ++j) { p->acur[slots[j]] ^= 1; p->audio_len[slots[j]] = new_len; }
  return MC_OK;
}

// The ragged counterpart (mc_pool_push_audio_ragged / mc_pool_push_pcm_ragged) for contexts of different length.
template <typename Stage>
int pool_encode_ragged(mc_pool* p, const int32_t* slots, int n, int len, int keep_frames, int64_t* codes_out, mc_stream_t stream_,
                       int kind, Stage stage) {
  mc_handle* h = p->h;
  MC_CUDA(h, cudaEventRecord(p->order_ev, (cudaStream_t)stream_));
  MC_CUDA(h, cudaStreamWaitEvent(p->own, p->order_ev, 0));
  cudaStream_t stream = p->own;
  const int hop = pool_hop(p);
  const int C = p->C, cap = p->cap_samples, rows = n * C, keep = keep_frames;
  const int T_max = pool_fill_ragged_table(p, slots, n, len, p->ctx_samples, p->audio_len, p->acur);
  const int F_max = (T_max + hop - 1) / hop;
  int F_min = F_max;
  for (int j = 0; j < n; ++j) F_min = std::min(F_min, (p->pin_table[4 * j + 3] + hop - 1) / hop);
  const int cut = ragged_cut(F_max - F_min + keep, F_max);
  const RaggedKeep rg{p->dev_table, C, keep};
  auto body = [&]() -> int {
    MC_CUDA(h, cudaMemcpyAsync(p->dev_table, p->pin_table, (size_t)n * 16, cudaMemcpyHostToDevice, stream));
    MC_TRY(stage(stream));
    pool_roll_ragged_kernel<float><<<dim3((T_max + 255) / 256, rows), 256, 0, stream>>>(p->dev_table, C, cap, len, p->audio[0], p->audio[1],
                                                                                       p->dev_chunk, p->batch_audio, cap, T_max);
    MC_LAUNCH_CHECK(h, "pool_roll_ragged_kernel");
    MC_TRY(encode_impl(h, p->batch_audio, cap, rows, T_max, cut, p->dev_codes_out, nullptr, nullptr, stream, &rg));
    MC_CUDA(h, cudaMemcpyAsync(p->pin_codes_out, p->dev_codes_out, (size_t)rows * keep * 8, cudaMemcpyDeviceToHost, stream));
    return MC_OK;
  };
  MC_TRY(run_or_replay(p, std::make_tuple(kind, T_max, len, cut, n, keep), stream, body));
  MC_CUDA(h, cudaStreamSynchronize(stream));
  memcpy(codes_out, p->pin_codes_out, (size_t)rows * keep * 8);
  for (int j = 0; j < n; ++j) { p->acur[slots[j]] ^= 1; p->audio_len[slots[j]] = p->pin_table[4 * j + 3]; }
  return MC_OK;
}

// mc_pool_push_audio's staging: the chunks go through pinned memory and one 2-D copy.
void pool_stage_chunks_host(mc_pool* p, const float* chunks, int rows, int len) {
  for (int r = 0; r < rows; ++r) memcpy(p->pin_chunk + (size_t)r * p->cap_samples, chunks + (size_t)r * len, (size_t)len * 4);
}
int pool_stage_chunks_device(mc_pool* p, int rows, int len, cudaStream_t stream) {
  const size_t pitch = (size_t)p->cap_samples * 4;
  MC_CUDA(p->h, cudaMemcpy2DAsync(p->dev_chunk, pitch, p->pin_chunk, pitch, (size_t)len * 4, rows, cudaMemcpyHostToDevice, stream));
  return MC_OK;
}
}  // namespace

extern "C" {

int mc_pool_destroy(mc_pool* p) {
  if (!p) return MC_OK;
  pool_drop_graphs(p);
  pool_free_emit(p);
  for (int i = 0; i < 2; ++i) { if (p->audio[i]) cudaFree(p->audio[i]); if (p->codes[i]) cudaFree(p->codes[i]); }
  for (void* d : {(void*)p->dev_chunk, (void*)p->batch_audio, (void*)p->dev_codes_in, (void*)p->batch_codes, (void*)p->dev_table,
                  (void*)p->dev_codes_out, (void*)p->dev_wav_out})
    if (d) cudaFree(d);
  for (void* q : {(void*)p->pin_chunk, (void*)p->pin_codes_in, (void*)p->pin_table, (void*)p->pin_codes_out, (void*)p->pin_wav_out})
    if (q) cudaFreeHost(q);
  for (auto& r : p->resamplers) cudaFree(r.taps);
  if (p->pin_pcm) cudaFreeHost(p->pin_pcm);
  if (p->pin_items) cudaFreeHost(p->pin_items);
  if (p->order_ev) cudaEventDestroy(p->order_ev);
  if (p->own) cudaStreamDestroy(p->own);
  delete p;
  return MC_OK;
}

int mc_pool_create(mc_handle* h, int32_t channels, int32_t context_samples, int32_t max_chunk_samples, int32_t max_sessions,
                   mc_pool** out) {
  MC_ENTER(h);
  if (!out || channels < 1 || context_samples < 1 || max_sessions < 1) return h->fail(MC_ERR_ARG, "mc_pool_create: bad arguments");
  int hop = 1;
  for (int i = 0; i < h->spec.n_convs; ++i) hop *= h->spec.conv_strides[i];
  mc_pool* p = new mc_pool();
  p->h = h; p->C = channels; p->max_sessions = max_sessions;
  p->ctx_samples = context_samples;
  p->ctx_frames = context_samples / hop;
  p->cap_samples = std::max(context_samples, max_chunk_samples);
  p->cap_frames = (p->cap_samples + hop - 1) / hop;
  if (p->cap_frames > h->spec.max_positions) { delete p; return h->fail(MC_ERR_ARG, "mc_pool_create: context exceeds RoPE table"); }
  p->audio_len.assign(max_sessions, 0); p->code_len.assign(max_sessions, 0);
  p->acur.assign(max_sessions, 0); p->ccur.assign(max_sessions, 0);
  p->emit_has_prev.assign(max_sessions, 0);
  const size_t rows = (size_t)max_sessions * channels;
  const size_t ab = rows * p->cap_samples * 4, cb = rows * p->cap_frames * 8;
  const size_t wb = rows * p->cap_frames * hop * 4;   // decoded windows: up to cap_frames * hop >= cap_samples samples each
  cudaError_t e = cudaSuccess;
  auto dev = [&](void** q, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(q, bytes); };
  auto pin = [&](void** q, size_t bytes) { if (e == cudaSuccess) e = cudaMallocHost(q, bytes); };
  for (int i = 0; i < 2; ++i) { dev((void**)&p->audio[i], ab); dev((void**)&p->codes[i], cb); }
  dev((void**)&p->dev_chunk, ab); dev((void**)&p->batch_audio, ab); dev((void**)&p->dev_wav_out, wb);
  dev((void**)&p->dev_codes_in, cb); dev((void**)&p->batch_codes, cb); dev((void**)&p->dev_codes_out, cb);
  dev((void**)&p->dev_table, (size_t)max_sessions * 16);
  pin((void**)&p->pin_chunk, ab); pin((void**)&p->pin_wav_out, wb);
  pin((void**)&p->pin_codes_in, cb); pin((void**)&p->pin_codes_out, cb);
  pin((void**)&p->pin_table, (size_t)max_sessions * 16);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->own, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->order_ev, cudaEventDisableTiming);
  if (e != cudaSuccess) { mc_pool_destroy(p); return h->fail(MC_ERR_NOMEM, "mc_pool_create: %s", cudaGetErrorString(e)); }
  *out = p;
  return MC_OK;
}

int mc_pool_reset(mc_pool* p, int32_t slot, int32_t audio, int32_t codes) {
  if (!p || slot < 0 || slot >= p->max_sessions) return MC_ERR_ARG;
  if (audio) p->audio_len[slot] = 0;
  if (codes) { p->code_len[slot] = 0; p->emit_has_prev[slot] = 0; }
  return MC_OK;
}

int mc_pool_context_len(mc_pool* p, int32_t slot, int32_t* audio_len, int32_t* code_len) {
  if (!p || slot < 0 || slot >= p->max_sessions) return MC_ERR_ARG;
  if (audio_len) *audio_len = p->audio_len[slot];
  if (code_len) *code_len = p->code_len[slot];
  return MC_OK;
}

int mc_pool_set_graphs(mc_pool* p, int32_t enabled) {
  if (!p) return MC_ERR_ARG;
  p->use_graphs = enabled != 0;
  if (!enabled) pool_drop_graphs(p);
  return MC_OK;
}

/* chunks: HOST fp32 [n][C][len]; codes_out: HOST int64 [n][C][keep] (keep = keep_frames, or every frame when 0). */
int mc_pool_push_audio(mc_pool* p, const int32_t* slots, int32_t n, const float* chunks, int32_t len, int32_t keep_frames,
                       int64_t* codes_out, int32_t* frames_out, mc_stream_t stream_) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  int old_len = 0;
  MC_TRY(pool_check_slots(p, slots, n, p->audio_len, &old_len, "mc_pool_push_audio"));
  if (!chunks || !codes_out || len < 1) return h->fail(MC_ERR_ARG, "mc_pool_push_audio: bad arguments");
  if (len > p->cap_samples) return h->fail(MC_ERR_ARG, "mc_pool_push_audio: chunk of %d samples exceeds the capacity %d", len, p->cap_samples);
  const int rows = n * p->C;
  pool_stage_chunks_host(p, chunks, rows, len);
  return pool_encode_uniform(p, slots, n, old_len, len, keep_frames, codes_out, frames_out, stream_, 0,
                             [&](cudaStream_t st) { return pool_stage_chunks_device(p, rows, len, st); });
}

/* codes: HOST int64 [n][C][len]; wav_out: HOST fp32 [n][C][keep] (keep = keep_samples, or the whole window when 0). */
int mc_pool_push_codes(mc_pool* p, const int32_t* slots, int32_t n, const int64_t* codes, int32_t len, int32_t keep_samples,
                       float* wav_out, int32_t* samples_out, mc_stream_t stream_) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  int old_len = 0;
  MC_TRY(pool_check_slots(p, slots, n, p->code_len, &old_len, "mc_pool_push_codes"));
  if (!codes || !wav_out || len < 1) return h->fail(MC_ERR_ARG, "mc_pool_push_codes: bad arguments");
  if (len > p->cap_frames) return h->fail(MC_ERR_ARG, "mc_pool_push_codes: %d frames exceed the capacity %d", len, p->cap_frames);
  MC_CUDA(h, cudaEventRecord(p->order_ev, (cudaStream_t)stream_));
  MC_CUDA(h, cudaStreamWaitEvent(p->own, p->order_ev, 0));
  cudaStream_t stream = p->own;
  int hop = 1;
  for (int i = 0; i < h->spec.n_convs; ++i) hop *= h->spec.conv_strides[i];
  const int C = p->C, cap = p->cap_frames, rows = n * C;
  const int new_len = std::min(old_len + len, std::max(len, p->ctx_frames));
  const int keep_old = new_len - len;
  const int total = new_len * hop;
  const int keep = (keep_samples <= 0 || keep_samples > total) ? total : keep_samples;
  for (int r = 0; r < rows; ++r) memcpy(p->pin_codes_in + (size_t)r * cap, codes + (size_t)r * len, (size_t)len * 8);
  for (int j = 0; j < n; ++j) { p->pin_table[2 * j] = slots[j]; p->pin_table[2 * j + 1] = p->ccur[slots[j]]; }
  auto body = [&]() -> int {
    MC_CUDA(h, cudaMemcpyAsync(p->dev_table, p->pin_table, (size_t)n * 8, cudaMemcpyHostToDevice, stream));
    MC_CUDA(h, cudaMemcpy2DAsync(p->dev_codes_in, (size_t)cap * 8, p->pin_codes_in, (size_t)cap * 8, (size_t)len * 8, rows, cudaMemcpyHostToDevice, stream));
    pool_roll_kernel<long long><<<dim3((new_len + 255) / 256, rows), 256, 0, stream>>>(
        p->dev_table, C, cap, old_len, keep_old, len, reinterpret_cast<long long*>(p->codes[0]), reinterpret_cast<long long*>(p->codes[1]),
        reinterpret_cast<const long long*>(p->dev_codes_in), reinterpret_cast<long long*>(p->batch_codes), new_len);
    MC_LAUNCH_CHECK(h, "pool_roll_kernel");
    MC_TRY(decode_impl(h, p->batch_codes, nullptr, rows, new_len, keep, p->dev_wav_out, stream));
    MC_CUDA(h, cudaMemcpyAsync(p->pin_wav_out, p->dev_wav_out, (size_t)rows * keep * 4, cudaMemcpyDeviceToHost, stream));
    return MC_OK;
  };
  MC_TRY(run_or_replay(p, std::make_tuple(1, old_len, len, keep, n, 0), stream, body));
  MC_CUDA(h, cudaStreamSynchronize(stream));
  memcpy(wav_out, p->pin_wav_out, (size_t)rows * keep * 4);
  if (samples_out) *samples_out = keep;
  for (int j = 0; j < n; ++j) { p->ccur[slots[j]] ^= 1; p->code_len[slots[j]] = new_len; }
  return MC_OK;
}

/* The emit chain of mc_stream_set_emit, shared by every slot of the pool; every slot forgets its previous chunk. */
int mc_pool_set_emit(mc_pool* p, int32_t chunk_samples, int32_t fade_samples, float target_rms, float silence_rms_threshold,
                     const float* fade_in) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  if (chunk_samples < 1 || fade_samples < 1 || fade_samples > chunk_samples || !fade_in)
    return h->fail(MC_ERR_ARG, "mc_pool_set_emit: need 0 < fade (%d) <= chunk (%d) and a ramp", fade_samples, chunk_samples);
  if (chunk_samples + fade_samples > p->cap_samples)
    return h->fail(MC_ERR_ARG, "mc_pool_set_emit: chunk + fade exceeds the session capacity %d", p->cap_samples);
  MC_CUDA(h, cudaStreamSynchronize(p->own));
  pool_drop_graphs(p);   // the captured kernels carry the old parameters and buffers
  pool_free_emit(p);
  std::fill(p->emit_has_prev.begin(), p->emit_has_prev.end(), 0);
  const size_t fb = (size_t)fade_samples * 4;
  cudaError_t e = cudaMalloc(&p->emit_fade_in, fb);
  if (e == cudaSuccess) e = cudaMalloc(&p->emit_prev_tails, fb * p->max_sessions);
  if (e == cudaSuccess) e = cudaMallocHost(&p->pin_emit, (size_t)p->max_sessions * (2 * chunk_samples + fade_samples) * 4);
  if (e == cudaSuccess) e = cudaMemcpy(p->emit_fade_in, fade_in, fb, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(p->emit_prev_tails, 0, fb * p->max_sessions);
  if (e != cudaSuccess) { pool_free_emit(p); return h->fail(MC_ERR_NOMEM, "mc_pool_set_emit: %s", cudaGetErrorString(e)); }
  p->emit_chunk = chunk_samples; p->emit_fade = fade_samples;
  p->emit_target_rms = target_rms; p->emit_silence_thr = silence_rms_threshold;
  return MC_OK;
}

/* mc_stream_push_codes_emit for n sessions in one launch.  codes: HOST int64 [n][len]; out: HOST fp32 [n][2*chunk + fade],
 * item j in the layout of mc_stream_push_codes_emit.  Every slot of one call must be at the same point of its stream:
 * all first chunks (empty code context) or all continuing ones. */
int mc_pool_push_codes_emit(mc_pool* p, const int32_t* slots, int32_t n, const int64_t* codes, int32_t len, float* out,
                            int32_t* had_prev, mc_stream_t stream_) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  int old_len = 0;
  MC_TRY(pool_check_slots(p, slots, n, p->code_len, &old_len, "mc_pool_push_codes_emit"));
  if (!codes || !out || len < 1) return h->fail(MC_ERR_ARG, "mc_pool_push_codes_emit: bad arguments");
  if (len > p->cap_frames) return h->fail(MC_ERR_ARG, "mc_pool_push_codes_emit: %d frames exceed the capacity %d", len, p->cap_frames);
  if (p->C != 1) return h->fail(MC_ERR_ARG, "mc_pool_push_codes_emit: the emit chain is mono (pad_or_trim rejects [C,T])");
  if (p->emit_chunk <= 0) return h->fail(MC_ERR_STATE, "mc_pool_push_codes_emit: call mc_pool_set_emit first");
  int hop = 1;
  for (int i = 0; i < h->spec.n_convs; ++i) hop *= h->spec.conv_strides[i];
  const int chunk = p->emit_chunk, fade = p->emit_fade, cap = p->cap_frames;
  if (len * hop != chunk)
    return h->fail(MC_ERR_ARG, "mc_pool_push_codes_emit: %d codes decode to %d samples, chunk is %d", len, len * hop, chunk);
  const int new_len = std::min(old_len + len, std::max(len, p->ctx_frames));
  const int keep_old = new_len - len;
  const int keep = std::min(new_len * hop, chunk + fade);
  // the stream's rules (realtime_agent_v2.py:566-568) for every slot, before any work or state change
  for (int j = 0; j < n; ++j) {
    if (p->emit_has_prev[slots[j]] && keep != chunk + fade)
      return h->fail(MC_ERR_STATE, "mc_pool_push_codes_emit: slot %d: only %d decoded samples for chunk %d + fade %d", slots[j], keep,
                     chunk, fade);
    if (!p->emit_has_prev[slots[j]] && keep != chunk)
      return h->fail(MC_ERR_STATE, "mc_pool_push_codes_emit: slot %d: the first emitted chunk needs an empty code context (reset first)",
                     slots[j]);
  }
  const int has_prev = p->emit_has_prev[slots[0]];
  for (int j = 1; j < n; ++j)
    if (p->emit_has_prev[slots[j]] != has_prev)
      return h->fail(MC_ERR_ARG, "mc_pool_push_codes_emit: slots %d and %d mix a first chunk with a continuing one; batch them separately",
                     slots[0], slots[j]);
  MC_CUDA(h, cudaEventRecord(p->order_ev, (cudaStream_t)stream_));
  MC_CUDA(h, cudaStreamWaitEvent(p->own, p->order_ev, 0));
  cudaStream_t stream = p->own;
  const int block = 2 * chunk + fade;
  for (int j = 0; j < n; ++j) memcpy(p->pin_codes_in + (size_t)j * cap, codes + (size_t)j * len, (size_t)len * 8);
  for (int j = 0; j < n; ++j) { p->pin_table[2 * j] = slots[j]; p->pin_table[2 * j + 1] = p->ccur[slots[j]]; }
  auto body = [&]() -> int {
    MC_CUDA(h, cudaMemcpyAsync(p->dev_table, p->pin_table, (size_t)n * 8, cudaMemcpyHostToDevice, stream));
    MC_CUDA(h, cudaMemcpy2DAsync(p->dev_codes_in, (size_t)cap * 8, p->pin_codes_in, (size_t)cap * 8, (size_t)len * 8, n, cudaMemcpyHostToDevice, stream));
    pool_roll_kernel<long long><<<dim3((new_len + 255) / 256, n), 256, 0, stream>>>(
        p->dev_table, 1, cap, old_len, keep_old, len, reinterpret_cast<long long*>(p->codes[0]), reinterpret_cast<long long*>(p->codes[1]),
        reinterpret_cast<const long long*>(p->dev_codes_in), reinterpret_cast<long long*>(p->batch_codes), new_len);
    MC_LAUNCH_CHECK(h, "pool_roll_kernel");
    MC_TRY(decode_impl(h, p->batch_codes, nullptr, n, new_len, keep, p->dev_wav_out, stream));
    mc_launch(h, emit_chunk_pool_kernel, dim3(n), dim3(POST_THREADS), 0, stream, (const float*)p->dev_wav_out, (long long)keep, keep,
              (const int*)p->dev_table, chunk, fade, has_prev, p->emit_target_rms, p->emit_silence_thr, (const float*)p->emit_fade_in,
              p->emit_prev_tails, p->pin_emit);                  // the blocks land in pinned host memory directly
    MC_LAUNCH_CHECK(h, "emit_chunk_pool_kernel");
    return MC_OK;
  };
  MC_TRY(run_or_replay(p, std::make_tuple(2 + has_prev, old_len, len, keep, n, 0), stream, body));
  MC_CUDA(h, cudaStreamSynchronize(stream));
  memcpy(out, p->pin_emit, (size_t)n * block * 4);
  if (had_prev) *had_prev = has_prev;
  for (int j = 0; j < n; ++j) { p->ccur[slots[j]] ^= 1; p->code_len[slots[j]] = new_len; p->emit_has_prev[slots[j]] = 1; }
  return MC_OK;
}

// ---- ragged batches: the sessions of one call may hold contexts of different length (a stream in its warm-up next to
// ones in steady state).  Equal lengths take the uniform call above; different lengths need causal attention.
namespace {
int pool_ragged_causal(mc_pool* p, const char* what) {
  if (p->h->spec.window_right != 0)
    return p->h->fail(MC_ERR_ARG, "%s: contexts of different length need causal attention (window_right = %d); batch them separately",
                      what, p->h->spec.window_right);
  return MC_OK;
}
}  // namespace

int mc_pool_push_audio_ragged(mc_pool* p, const int32_t* slots, int32_t n, const float* chunks, int32_t len, int32_t keep_frames,
                              int64_t* codes_out, mc_stream_t stream_) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  int common = 0;
  MC_TRY(pool_check_slots(p, slots, n, p->audio_len, &common, "mc_pool_push_audio_ragged", false));
  if (!chunks || !codes_out || len < 1) return h->fail(MC_ERR_ARG, "mc_pool_push_audio_ragged: bad arguments");
  if (len > p->cap_samples)
    return h->fail(MC_ERR_ARG, "mc_pool_push_audio_ragged: chunk of %d samples exceeds the capacity %d", len, p->cap_samples);
  const int hop = pool_hop(p);
  if (keep_frames < 1 || keep_frames > (len + hop - 1) / hop)
    return h->fail(MC_ERR_ARG, "mc_pool_push_audio_ragged: keep_frames %d outside 1..%d", keep_frames, (len + hop - 1) / hop);
  if (common >= 0) return mc_pool_push_audio(p, slots, n, chunks, len, keep_frames, codes_out, nullptr, stream_);
  MC_TRY(pool_ragged_causal(p, "mc_pool_push_audio_ragged"));
  const int rows = n * p->C;
  pool_stage_chunks_host(p, chunks, rows, len);
  return pool_encode_ragged(p, slots, n, len, keep_frames, codes_out, stream_, 4,
                            [&](cudaStream_t st) { return pool_stage_chunks_device(p, rows, len, st); });
}

int mc_pool_push_codes_ragged(mc_pool* p, const int32_t* slots, int32_t n, const int64_t* codes, int32_t len, int32_t keep_samples,
                              float* wav_out, int32_t* samples_out, mc_stream_t stream_) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  int common = 0;
  MC_TRY(pool_check_slots(p, slots, n, p->code_len, &common, "mc_pool_push_codes_ragged", false));
  if (!codes || !wav_out || !samples_out || len < 1) return h->fail(MC_ERR_ARG, "mc_pool_push_codes_ragged: bad arguments");
  if (len > p->cap_frames) return h->fail(MC_ERR_ARG, "mc_pool_push_codes_ragged: %d frames exceed the capacity %d", len, p->cap_frames);
  int hop = 1;
  for (int i = 0; i < h->spec.n_convs; ++i) hop *= h->spec.conv_strides[i];
  if (keep_samples < 1 || keep_samples > p->cap_frames * hop)
    return h->fail(MC_ERR_ARG, "mc_pool_push_codes_ragged: keep_samples %d outside 1..%d", keep_samples, p->cap_frames * hop);
  const int C = p->C, rows = n * C;
  if (common >= 0) {
    int got = 0;
    MC_TRY(mc_pool_push_codes(p, slots, n, codes, len, keep_samples, wav_out, &got, stream_));
    for (int r = rows - 1; r >= 1 && got < keep_samples; --r)    // rows of `got` samples -> rows of keep_samples, back to front
      memmove(wav_out + (size_t)r * keep_samples, wav_out + (size_t)r * got, (size_t)got * 4);
    for (int r = 0; r < rows && got < keep_samples; ++r)
      memset(wav_out + (size_t)r * keep_samples + got, 0, (size_t)(keep_samples - got) * 4);
    for (int j = 0; j < n; ++j) samples_out[j] = got;
    return MC_OK;
  }
  MC_TRY(pool_ragged_causal(p, "mc_pool_push_codes_ragged"));
  MC_CUDA(h, cudaEventRecord(p->order_ev, (cudaStream_t)stream_));
  MC_CUDA(h, cudaStreamWaitEvent(p->own, p->order_ev, 0));
  cudaStream_t stream = p->own;
  const int cap = p->cap_frames;
  const int F_max = pool_fill_ragged_table(p, slots, n, len, p->ctx_frames, p->code_len, p->ccur);
  int cut = 0, dec_keep = 0;
  ragged_decode_cut(p, n, F_max, hop, keep_samples, &cut, &dec_keep);
  for (int r = 0; r < rows; ++r) memcpy(p->pin_codes_in + (size_t)r * cap, codes + (size_t)r * len, (size_t)len * 8);
  auto body = [&]() -> int {
    MC_CUDA(h, cudaMemcpyAsync(p->dev_table, p->pin_table, (size_t)n * 16, cudaMemcpyHostToDevice, stream));
    MC_CUDA(h, cudaMemcpy2DAsync(p->dev_codes_in, (size_t)cap * 8, p->pin_codes_in, (size_t)cap * 8, (size_t)len * 8, rows, cudaMemcpyHostToDevice, stream));
    pool_roll_ragged_kernel<long long><<<dim3((F_max + 255) / 256, rows), 256, 0, stream>>>(
        p->dev_table, C, cap, len, reinterpret_cast<long long*>(p->codes[0]), reinterpret_cast<long long*>(p->codes[1]),
        reinterpret_cast<const long long*>(p->dev_codes_in), reinterpret_cast<long long*>(p->batch_codes), F_max, F_max);
    MC_LAUNCH_CHECK(h, "pool_roll_ragged_kernel");
    MC_TRY(decode_impl(h, p->batch_codes, nullptr, rows, F_max, dec_keep, p->dev_wav_out, stream));
    pool_gather_samples_ragged_kernel<<<dim3((keep_samples + 255) / 256, rows), 256, 0, stream>>>(
        p->dev_wav_out, dec_keep, p->dev_table, C, F_max * hop, hop, keep_samples, p->pin_wav_out);   // straight into pinned host memory
    MC_LAUNCH_CHECK(h, "pool_gather_samples_ragged_kernel");
    return MC_OK;
  };
  MC_TRY(run_or_replay(p, std::make_tuple(5, F_max, len, cut, n, keep_samples), stream, body));
  MC_CUDA(h, cudaStreamSynchronize(stream));
  memcpy(wav_out, p->pin_wav_out, (size_t)rows * keep_samples * 4);
  for (int j = 0; j < n; ++j) {
    samples_out[j] = std::min(keep_samples, p->pin_table[4 * j + 3] * hop);
    p->ccur[slots[j]] ^= 1;
    p->code_len[slots[j]] = p->pin_table[4 * j + 3];
  }
  return MC_OK;
}

int mc_pool_push_codes_emit_ragged(mc_pool* p, const int32_t* slots, int32_t n, const int64_t* codes, int32_t len, float* out,
                                   int32_t* had_prev, mc_stream_t stream_) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  int common = 0;
  MC_TRY(pool_check_slots(p, slots, n, p->code_len, &common, "mc_pool_push_codes_emit_ragged", false));
  if (!codes || !out || !had_prev || len < 1) return h->fail(MC_ERR_ARG, "mc_pool_push_codes_emit_ragged: bad arguments");
  if (len > p->cap_frames)
    return h->fail(MC_ERR_ARG, "mc_pool_push_codes_emit_ragged: %d frames exceed the capacity %d", len, p->cap_frames);
  if (p->C != 1) return h->fail(MC_ERR_ARG, "mc_pool_push_codes_emit_ragged: the emit chain is mono (pad_or_trim rejects [C,T])");
  if (p->emit_chunk <= 0) return h->fail(MC_ERR_STATE, "mc_pool_push_codes_emit_ragged: call mc_pool_set_emit first");
  int hop = 1;
  for (int i = 0; i < h->spec.n_convs; ++i) hop *= h->spec.conv_strides[i];
  const int chunk = p->emit_chunk, fade = p->emit_fade, cap = p->cap_frames;
  if (len * hop != chunk)
    return h->fail(MC_ERR_ARG, "mc_pool_push_codes_emit_ragged: %d codes decode to %d samples, chunk is %d", len, len * hop, chunk);
  // the stream's rules (realtime_agent_v2.py:566-568) for every slot, before any work or state change
  for (int j = 0; j < n; ++j) {
    const int keep = std::min(std::min(p->code_len[slots[j]] + len, std::max(len, p->ctx_frames)) * hop, chunk + fade);
    if (p->emit_has_prev[slots[j]] && keep != chunk + fade)
      return h->fail(MC_ERR_STATE, "mc_pool_push_codes_emit_ragged: slot %d: only %d decoded samples for chunk %d + fade %d", slots[j],
                     keep, chunk, fade);
    if (!p->emit_has_prev[slots[j]] && keep != chunk)
      return h->fail(MC_ERR_STATE, "mc_pool_push_codes_emit_ragged: slot %d: the first emitted chunk needs an empty code context (reset first)",
                     slots[j]);
  }
  if (common >= 0) {   // equal lengths: equal keeps, so the rules above leave one shared had_prev
    int hp = 0;
    MC_TRY(mc_pool_push_codes_emit(p, slots, n, codes, len, out, &hp, stream_));
    for (int j = 0; j < n; ++j) had_prev[j] = hp;
    return MC_OK;
  }
  MC_TRY(pool_ragged_causal(p, "mc_pool_push_codes_emit_ragged"));
  MC_CUDA(h, cudaEventRecord(p->order_ev, (cudaStream_t)stream_));
  MC_CUDA(h, cudaStreamWaitEvent(p->own, p->order_ev, 0));
  cudaStream_t stream = p->own;
  const int block = 2 * chunk + fade;
  const int F_max = pool_fill_ragged_table(p, slots, n, len, p->ctx_frames, p->code_len, p->ccur);
  int cut = 0, dec_keep = 0;
  ragged_decode_cut(p, n, F_max, hop, chunk + fade, &cut, &dec_keep);
  for (int j = 0; j < n; ++j) memcpy(p->pin_codes_in + (size_t)j * cap, codes + (size_t)j * len, (size_t)len * 8);
  auto body = [&]() -> int {
    MC_CUDA(h, cudaMemcpyAsync(p->dev_table, p->pin_table, (size_t)n * 16, cudaMemcpyHostToDevice, stream));
    MC_CUDA(h, cudaMemcpy2DAsync(p->dev_codes_in, (size_t)cap * 8, p->pin_codes_in, (size_t)cap * 8, (size_t)len * 8, n, cudaMemcpyHostToDevice, stream));
    pool_roll_ragged_kernel<long long><<<dim3((F_max + 255) / 256, n), 256, 0, stream>>>(
        p->dev_table, 1, cap, len, reinterpret_cast<long long*>(p->codes[0]), reinterpret_cast<long long*>(p->codes[1]),
        reinterpret_cast<const long long*>(p->dev_codes_in), reinterpret_cast<long long*>(p->batch_codes), F_max, F_max);
    MC_LAUNCH_CHECK(h, "pool_roll_ragged_kernel");
    MC_TRY(decode_impl(h, p->batch_codes, nullptr, n, F_max, dec_keep, p->dev_wav_out, stream));
    mc_launch(h, emit_chunk_pool_ragged_kernel, dim3(n), dim3(POST_THREADS), 0, stream, (const float*)p->dev_wav_out, (long long)dec_keep,
              (const int*)p->dev_table, F_max * hop, hop, chunk, fade, p->emit_target_rms, p->emit_silence_thr,
              (const float*)p->emit_fade_in, p->emit_prev_tails, p->pin_emit);   // the blocks land in pinned host memory directly
    MC_LAUNCH_CHECK(h, "emit_chunk_pool_ragged_kernel");
    return MC_OK;
  };
  MC_TRY(run_or_replay(p, std::make_tuple(6, F_max, len, cut, n, 0), stream, body));
  MC_CUDA(h, cudaStreamSynchronize(stream));
  memcpy(out, p->pin_emit, (size_t)n * block * 4);
  for (int j = 0; j < n; ++j) {
    had_prev[j] = p->emit_has_prev[slots[j]];
    p->ccur[slots[j]] ^= 1;
    p->code_len[slots[j]] = p->pin_table[4 * j + 3];
    p->emit_has_prev[slots[j]] = 1;
  }
  return MC_OK;
}

int mc_pool_graph_count(mc_pool* p, int32_t* keys, int32_t* captured) {
  if (!p) return MC_ERR_ARG;
  int c = 0;
  for (const auto& kv : p->graphs) c += kv.second.exec != nullptr;
  if (keys) *keys = (int32_t)p->graphs.size();
  if (captured) *captured = c;
  return MC_OK;
}

int mc_pool_read_audio(mc_pool* p, int32_t slot, float* out_host, int32_t n) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  if (slot < 0 || slot >= p->max_sessions || !out_host || n < 1 || n > p->audio_len[slot])
    return h->fail(MC_ERR_ARG, "mc_pool_read_audio: need a slot < %d and 1 <= n <= its %d context samples", p->max_sessions,
                   (slot >= 0 && slot < p->max_sessions) ? p->audio_len[slot] : 0);
  const size_t cap = (size_t)p->cap_samples;
  const float* src = p->audio[p->acur[slot]] + (size_t)slot * p->C * cap + (p->audio_len[slot] - n);
  MC_CUDA(h, cudaMemcpy2DAsync(out_host, (size_t)n * 4, src, cap * 4, (size_t)n * 4, p->C, cudaMemcpyDeviceToHost, p->own));
  MC_CUDA(h, cudaStreamSynchronize(p->own));
  return MC_OK;
}

}  // extern "C"

// ---- live-stream ingest: pooled sessions whose clients send s16 / f32 PCM at their own rate, [C_in][n] per chunk
// (what AudioTokenizer._prep_audio_for_tokenization does on the host: int16 / 32768, the mean over channels for a mono
// codec, the polyphase resampler), converted and resampled by pool_ingest_kernel inside the push's graph.
namespace {
size_t align16(size_t b) { return (b + 15) & ~(size_t)15; }
size_t pcm_item_bytes(const mc_pcm_chunk& it) { return align16((size_t)it.channels_in * it.n_in * (it.format == PCM_S16 ? 2 : 4)); }

// (Re)allocate the pinned payload staging.  The pcm graphs bake its address in, so they go; every other graph stays.
int pool_pcm_alloc(mc_pool* p, size_t bytes, const char* what) {
  mc_handle* h = p->h;
  MC_CUDA(h, cudaStreamSynchronize(p->own));
  for (auto it = p->graphs.begin(); it != p->graphs.end();) {
    if (std::get<0>(it->first) >= 7) {
      if (it->second.exec) cudaGraphExecDestroy(it->second.exec);
      it = p->graphs.erase(it);
    } else {
      ++it;
    }
  }
  if (p->pin_pcm) cudaFreeHost(p->pin_pcm);
  p->pin_pcm = nullptr;
  p->pin_pcm_bytes = 0;
  cudaError_t e = cudaSuccess;
  if (!p->pin_items) e = cudaMallocHost(&p->pin_items, (size_t)p->max_sessions * sizeof(PoolIngestItem));
  if (e == cudaSuccess) e = cudaMallocHost(&p->pin_pcm, bytes);
  if (e != cudaSuccess) { p->pin_pcm = nullptr; return h->fail(MC_ERR_NOMEM, "%s: %s", what, cudaGetErrorString(e)); }
  p->pin_pcm_bytes = bytes;
  return MC_OK;
}

const mc_pool::Resampler* pool_find_resampler(const mc_pool* p, int sr) {
  for (const auto& r : p->resamplers)
    if (r.sr == sr) return &r;
  return nullptr;
}

// Every check of a pcm push's items, before any work or state change.
int pool_check_pcm(mc_pool* p, int n, const mc_pcm_chunk* items, const void* payload, int len, const char* what) {
  mc_handle* h = p->h;
  if (!items || !payload || len < 1) return h->fail(MC_ERR_ARG, "%s: bad arguments", what);
  if (len > p->cap_samples) return h->fail(MC_ERR_ARG, "%s: chunk of %d samples exceeds the capacity %d", what, len, p->cap_samples);
  for (int j = 0; j < n; ++j) {
    const mc_pcm_chunk& it = items[j];
    if (it.format != PCM_S16 && it.format != PCM_F32)
      return h->fail(MC_ERR_ARG, "%s: item %d: format %d (only MC_PCM_S16 and MC_PCM_F32)", what, j, it.format);
    if (p->C > 1 && it.channels_in != p->C)
      return h->fail(MC_ERR_ARG, "%s: item %d: %d channels for a %d-channel pool", what, j, it.channels_in, p->C);
    if (p->C == 1 && (it.channels_in < 1 || it.channels_in > MC_POOL_MAX_MIX_CHANNELS))
      return h->fail(MC_ERR_ARG, "%s: item %d: %d channels (a mono pool mixes 1..%d)", what, j, it.channels_in, MC_POOL_MAX_MIX_CHANNELS);
    if (it.n_in < 1 || it.offset_bytes < 0 || (it.channels_in > 1 && it.ld < it.n_in))
      return h->fail(MC_ERR_ARG, "%s: item %d: bad layout (n_in %d, ld %lld, offset %lld)", what, j, it.n_in, (long long)it.ld,
                     (long long)it.offset_bytes);
    if (p->pcm_max_in > 0 && (it.n_in > p->pcm_max_in || it.channels_in > p->pcm_max_channels))
      return h->fail(MC_ERR_ARG, "%s: item %d: %d x %d samples exceed the staging reserved for %d x %d", what, j, it.channels_in, it.n_in,
                     p->pcm_max_channels, p->pcm_max_in);
    long long n_out = it.n_in;
    if (it.sample_rate != h->spec.sample_rate) {
      const mc_pool::Resampler* r = pool_find_resampler(p, it.sample_rate);
      if (!r) return h->fail(MC_ERR_ARG, "%s: item %d: no resampler registered for %d Hz", what, j, it.sample_rate);
      n_out = ((long long)it.n_in * r->up + r->down - 1) / r->down;
    }
    if (n_out != len)
      return h->fail(MC_ERR_ARG, "%s: item %d: %d samples at %d Hz resample to %lld, the call's length is %d", what, j, it.n_in,
                     it.sample_rate, n_out, len);
  }
  return MC_OK;
}

// Copy the items' rows into the pinned staging and fill the kernel's table.  Unless mc_pool_reserve_pcm fixed the staging,
// it grows when a call needs more, to room for every slot at the call's largest item, so sessions that join do not
// reallocate it (and drop the pcm graphs) again.
int pool_stage_pcm_host(mc_pool* p, int n, const mc_pcm_chunk* items, const void* payload, const char* what) {
  size_t total = 0, largest = 0;
  for (int j = 0; j < n; ++j) { total += pcm_item_bytes(items[j]); largest = std::max(largest, pcm_item_bytes(items[j])); }
  if (total > p->pin_pcm_bytes || !p->pin_items)
    MC_TRY(pool_pcm_alloc(p, std::max(largest * p->max_sessions, 2 * p->pin_pcm_bytes), what));
  size_t off = 0;
  for (int j = 0; j < n; ++j) {
    const mc_pcm_chunk& it = items[j];
    const size_t es = it.format == PCM_S16 ? 2 : 4, row = (size_t)it.n_in * es;
    for (int c = 0; c < it.channels_in; ++c)
      memcpy(p->pin_pcm + off + c * row, static_cast<const unsigned char*>(payload) + it.offset_bytes + (size_t)c * it.ld * es, row);
    PoolIngestItem& d = p->pin_items[j];
    const mc_pool::Resampler* r = it.sample_rate != p->h->spec.sample_rate ? pool_find_resampler(p, it.sample_rate) : nullptr;
    d.taps = r ? r->taps : nullptr;
    d.offset = (long long)off;
    d.pre_remove = r ? r->pre_remove : 0;
    d.format = it.format; d.channels = it.channels_in; d.n_in = it.n_in;
    d.up = r ? r->up : 1; d.down = r ? r->down : 1; d.n_taps = r ? r->n_taps : 0;
    off += pcm_item_bytes(it);
  }
  return MC_OK;
}

int pool_stage_pcm_device(mc_pool* p, int n, int len, cudaStream_t stream) {
  pool_ingest_kernel<<<dim3((len + INGEST_TILE - 1) / INGEST_TILE, n * p->C), 256, 0, stream>>>(p->pin_items, p->pin_pcm, p->C, len,
                                                                                                  p->dev_chunk, p->cap_samples);
  MC_LAUNCH_CHECK(p->h, "pool_ingest_kernel");
  return MC_OK;
}
}  // namespace

extern "C" {

int mc_pool_set_resampler(mc_pool* p, int32_t sr_in, int32_t up, int32_t down, const float* taps, int32_t n_taps, int64_t pre_remove) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  const int sr = h->spec.sample_rate;
  if (sr_in < 1 || sr_in == sr || up < 1 || down < 1 || (int64_t)sr_in * up != (int64_t)sr * down || !taps || n_taps < 1 || pre_remove < 0)
    return h->fail(MC_ERR_ARG, "mc_pool_set_resampler: bad plan (%d Hz -> %d Hz, up %d, down %d, %d taps)", sr_in, sr, up, down, n_taps);
  if (ingest_span(up, down, n_taps) > INGEST_SPAN)
    return h->fail(MC_ERR_ARG, "mc_pool_set_resampler: %d Hz: a tile reads %lld input samples, more than %d", sr_in,
                   ingest_span(up, down, n_taps), INGEST_SPAN);
  if (!pool_find_resampler(p, sr_in) && (int)p->resamplers.size() >= MC_POOL_MAX_RESAMPLERS)
    return h->fail(MC_ERR_ARG, "mc_pool_set_resampler: already %d input rates registered", MC_POOL_MAX_RESAMPLERS);
  float* d = nullptr;
  cudaError_t e = cudaMalloc(&d, (size_t)n_taps * 4);
  if (e == cudaSuccess) e = cudaMemcpy(d, taps, (size_t)n_taps * 4, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    if (d) cudaFree(d);
    return h->fail(MC_ERR_NOMEM, "mc_pool_set_resampler: %s", cudaGetErrorString(e));
  }
  MC_CUDA(h, cudaStreamSynchronize(p->own));   // a replaced plan's taps may still be read by the last push
  mc_pool::Resampler* r = const_cast<mc_pool::Resampler*>(pool_find_resampler(p, sr_in));
  if (!r) { p->resamplers.emplace_back(); r = &p->resamplers.back(); }
  if (r->taps) cudaFree(r->taps);
  r->sr = sr_in; r->up = up; r->down = down; r->n_taps = n_taps; r->pre_remove = pre_remove; r->taps = d;
  return MC_OK;
}

int mc_pool_reserve_pcm(mc_pool* p, int32_t max_in_samples, int32_t max_in_channels) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  const int ch_limit = p->C > 1 ? p->C : MC_POOL_MAX_MIX_CHANNELS;
  if (max_in_samples < 1 || max_in_channels < 1 || max_in_channels > ch_limit)
    return h->fail(MC_ERR_ARG, "mc_pool_reserve_pcm: need max_in_samples >= 1 and 1 <= max_in_channels <= %d", ch_limit);
  const size_t bytes = (size_t)p->max_sessions * align16((size_t)max_in_samples * max_in_channels * 4);
  if (bytes != p->pin_pcm_bytes || !p->pin_items) MC_TRY(pool_pcm_alloc(p, bytes, "mc_pool_reserve_pcm"));
  p->pcm_max_in = max_in_samples;
  p->pcm_max_channels = max_in_channels;
  return MC_OK;
}

int mc_pool_push_pcm(mc_pool* p, const int32_t* slots, int32_t n, const mc_pcm_chunk* items, const void* payload, int32_t len,
                     int32_t keep_frames, int64_t* codes_out, int32_t* frames_out, mc_stream_t stream_) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  int old_len = 0;
  MC_TRY(pool_check_slots(p, slots, n, p->audio_len, &old_len, "mc_pool_push_pcm"));
  if (!codes_out) return h->fail(MC_ERR_ARG, "mc_pool_push_pcm: bad arguments");
  MC_TRY(pool_check_pcm(p, n, items, payload, len, "mc_pool_push_pcm"));
  MC_TRY(pool_stage_pcm_host(p, n, items, payload, "mc_pool_push_pcm"));
  return pool_encode_uniform(p, slots, n, old_len, len, keep_frames, codes_out, frames_out, stream_, 7,
                             [&](cudaStream_t st) { return pool_stage_pcm_device(p, n, len, st); });
}

int mc_pool_push_pcm_ragged(mc_pool* p, const int32_t* slots, int32_t n, const mc_pcm_chunk* items, const void* payload, int32_t len,
                            int32_t keep_frames, int64_t* codes_out, mc_stream_t stream_) {
  if (!p) return MC_ERR_ARG;
  mc_handle* h = p->h;
  MC_ENTER(h);
  int common = 0;
  MC_TRY(pool_check_slots(p, slots, n, p->audio_len, &common, "mc_pool_push_pcm_ragged", false));
  if (!codes_out) return h->fail(MC_ERR_ARG, "mc_pool_push_pcm_ragged: bad arguments");
  MC_TRY(pool_check_pcm(p, n, items, payload, len, "mc_pool_push_pcm_ragged"));
  const int hop = pool_hop(p);
  if (keep_frames < 1 || keep_frames > (len + hop - 1) / hop)
    return h->fail(MC_ERR_ARG, "mc_pool_push_pcm_ragged: keep_frames %d outside 1..%d", keep_frames, (len + hop - 1) / hop);
  if (common >= 0) return mc_pool_push_pcm(p, slots, n, items, payload, len, keep_frames, codes_out, nullptr, stream_);
  MC_TRY(pool_ragged_causal(p, "mc_pool_push_pcm_ragged"));
  MC_TRY(pool_stage_pcm_host(p, n, items, payload, "mc_pool_push_pcm_ragged"));
  return pool_encode_ragged(p, slots, n, len, keep_frames, codes_out, stream_, 8,
                            [&](cudaStream_t st) { return pool_stage_pcm_device(p, n, len, st); });
}

}  // extern "C"
