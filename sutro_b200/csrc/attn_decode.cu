// sutro_b200 — K2: paged-KV decode attention (one query token per sequence).
//
// HBM-bound: per generated token each sequence streams its whole K/V history
// once (ctx_len x 2 x hkv x 256 B per layer).  Design:
//   * grid = (kv_head, sequence); the G = hq/hkv query heads that share a KV
//     head are processed together so K/V are read from HBM exactly once (GQA).
//   * 4 warps per CTA; warp w owns KV pages w, w+4, ...  Each warp runs its own
//     kStages-deep ring of 8 KiB stages filled by cp.async.bulk (UBLKCP): one
//     lane issues a single flat 8 KiB copy per page (K tile + V tile of one
//     head are contiguous in the pool), completion arrives on an mbarrier.
//   * The pool stores tiles pre-swizzled (kernels.h), so the flat copy lands in
//     shared memory bank-conflict-free for ldmatrix / ldmatrix.trans.
//   * S = Q K^T and O += P V run on mma.sync m16n8k16 (bf16 in, fp32 acc) with
//     the G query heads as the (zero-padded) M rows; online softmax uses
//     quad-level warp shuffles; the 4 warps' partial (m, l, O) are merged
//     through shared memory at the end.
#include "common.cuh"
#include "kernels.h"

namespace sb {

namespace {

constexpr int kDecWarps = 4;
constexpr int kDecStages = 3;
constexpr int kStageBytes = 2 * kTileBytes;  // K tile + V tile = 8 KiB
constexpr int kDecSmem = kDecWarps * kDecStages * kStageBytes + 1024;
bool g_force_split = false;   // tests: exercise the 4-warp split kernel at any batch size
bool g_force_warp = false;    // tests: exercise the warp-per-pair kernel at any batch size

template <int G>
__global__ void __launch_bounds__(kDecWarps * 32)
attn_decode_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out,
                   const __nv_bfloat16* __restrict__ kv_layer,
                   const int32_t* __restrict__ page_table, int max_pages,
                   const int32_t* __restrict__ row_slot, const int32_t* __restrict__ ctx_len,
                   int hq, int hkv, float scale_log2) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~static_cast<uintptr_t>(127));
  __shared__ uint64_t full_bar[kDecWarps][kDecStages];
  __shared__ float red_m[kDecWarps][8];
  __shared__ float red_l[kDecWarps][8];

  const int kvh = blockIdx.x;
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int slot = row_slot[b];
  const int L = ctx_len[b];
  const int n_tiles = (L + kPageTokens - 1) / kPageTokens;
  const int32_t* pt = page_table + static_cast<size_t>(slot) * max_pages;

  uint8_t* my_smem = smem + warp * kDecStages * kStageBytes;
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kDecStages; ++s) mbar_init(smem_u32(&full_bar[warp][s]), 1);
    fence_mbar_init();
  }
  __syncwarp();

  auto issue = [&](int tile, int stage) {
    const int page = pt[tile];
    const __nv_bfloat16* src =
        kv_layer + (static_cast<size_t>(page) * hkv + kvh) * (2 * kTileElems);
    const uint32_t bar = smem_u32(&full_bar[warp][stage]);
    mbar_arrive_expect_tx(bar, kStageBytes);
    bulk_load_1d(smem_u32(my_smem + stage * kStageBytes), src, kStageBytes, bar);
  };

  // prologue: fill the ring
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kDecStages; ++s) {
      const int tile = warp + s * kDecWarps;
      if (tile < n_tiles) issue(tile, s);
    }
  }

  // Q fragments: rows = query heads of this KV group (row >= G is zero padding).
  const int ldq = (hq + 2 * hkv) * kHeadDim;
  const int qr = lane >> 2;
  uint32_t qa[8][2];  // [k-step][a0, a2]   (a1 = a3 = 0: rows 8..15 unused)
  {
    const __nv_bfloat16* qp =
        qkv + static_cast<size_t>(b) * ldq + (kvh * G + qr) * kHeadDim + 2 * (lane & 3);
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
      if (qr < G) {
        qa[kk][0] = *reinterpret_cast<const uint32_t*>(qp + kk * 16);
        qa[kk][1] = *reinterpret_cast<const uint32_t*>(qp + kk * 16 + 8);
      } else {
        qa[kk][0] = 0u;
        qa[kk][1] = 0u;
      }
    }
  }

  float o[16][2];  // rows 0..7 only (c0, c1 of each n-tile)
#pragma unroll
  for (int i = 0; i < 16; ++i) o[i][0] = o[i][1] = 0.f;
  float m_run = -INFINITY, l_run = 0.f;

  const int lm = lane >> 3;  // ldmatrix: which 8x8 matrix this lane addresses
  const int lr = lane & 7;

  int it = 0;
  for (int tile = warp; tile < n_tiles; tile += kDecWarps, ++it) {
    const int stage = it % kDecStages;
    const uint32_t phase = (it / kDecStages) & 1;
    mbar_wait(smem_u32(&full_bar[warp][stage]), phase);
    const uint32_t ks = smem_u32(my_smem + stage * kStageBytes);
    const uint32_t vs = ks + kTileBytes;

    // ---- S = Q K^T : 16 (padded heads) x 16 tokens ----
    float s0[4] = {0.f, 0.f, 0.f, 0.f};  // tokens 0..7
    float s1[4] = {0.f, 0.f, 0.f, 0.f};  // tokens 8..15
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
      const int tok = (lm >> 1) * 8 + lr;
      const int chunk = kk * 2 + (lm & 1);
      uint32_t b0, b1, b2, b3;
      ldmatrix_x4(ks + tok * 256 + ((chunk ^ (tok & 7)) << 4), b0, b1, b2, b3);
      const uint32_t a[4] = {qa[kk][0], 0u, qa[kk][1], 0u};
      mma_bf16_16816(s0, a, b0, b1);
      mma_bf16_16816(s1, a, b2, b3);
    }
    // ---- online softmax on row lane/4 (values c0, c1 of both n-tiles) ----
    const int tok0 = tile * kPageTokens + 2 * (lane & 3);
    float sv[4] = {s0[0], s0[1], s1[0], s1[1]};
    if (tok0 >= L) sv[0] = -INFINITY;
    if (tok0 + 1 >= L) sv[1] = -INFINITY;
    if (tok0 + 8 >= L) sv[2] = -INFINITY;
    if (tok0 + 9 >= L) sv[3] = -INFINITY;
    float mx = fmaxf(fmaxf(sv[0], sv[1]), fmaxf(sv[2], sv[3]));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    const float m_new = fmaxf(m_run, mx);  // finite: every visited tile has >= 1 valid token
    const float alpha = exp2f((m_run - m_new) * scale_log2);
    float p[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = exp2f((sv[i] - m_new) * scale_log2);
    float ps = p[0] + p[1] + p[2] + p[3];
    ps += __shfl_xor_sync(0xffffffffu, ps, 1);
    ps += __shfl_xor_sync(0xffffffffu, ps, 2);
    l_run = l_run * alpha + ps;
    m_run = m_new;
    const uint32_t pa[4] = {pack_bf16x2(p[0], p[1]), 0u, pack_bf16x2(p[2], p[3]), 0u};

    // ---- O = O * alpha + P V ----
#pragma unroll
    for (int nt = 0; nt < 16; nt += 2) {
      const int tok = (lm & 1) * 8 + lr;
      const int chunk = nt + (lm >> 1);
      uint32_t b0, b1, b2, b3;
      ldmatrix_x4_trans(vs + tok * 256 + ((chunk ^ (tok & 7)) << 4), b0, b1, b2, b3);
      float d0[4] = {o[nt][0] * alpha, o[nt][1] * alpha, 0.f, 0.f};
      float d1[4] = {o[nt + 1][0] * alpha, o[nt + 1][1] * alpha, 0.f, 0.f};
      mma_bf16_16816(d0, pa, b0, b1);
      mma_bf16_16816(d1, pa, b2, b3);
      o[nt][0] = d0[0];
      o[nt][1] = d0[1];
      o[nt + 1][0] = d1[0];
      o[nt + 1][1] = d1[1];
    }

    // ---- refill this stage with the tile kStages iterations ahead ----
    __syncwarp();
    const int next = tile + kDecStages * kDecWarps;
    if (lane == 0 && next < n_tiles) {
      fence_proxy_async_smem();  // generic-proxy reads above vs async-proxy write below
      issue(next, stage);
    }
  }

  // ---- merge the 4 warps' partial results ----
  __syncthreads();  // all bulk copies consumed; stage memory is reusable as scratch
  float* o_part = reinterpret_cast<float*>(smem) + warp * 8 * kHeadDim;  // [8][128] per warp
  if ((lane & 3) == 0) {
    red_m[warp][qr] = m_run;
    red_l[warp][qr] = l_run;
  }
#pragma unroll
  for (int nt = 0; nt < 16; ++nt) {
    float2* dst = reinterpret_cast<float2*>(o_part + qr * kHeadDim + nt * 8 + 2 * (lane & 3));
    *dst = make_float2(o[nt][0], o[nt][1]);
  }
  __syncthreads();
  {
    const int dim = threadIdx.x;  // 128 threads == 128 dims
    const float* o_all = reinterpret_cast<const float*>(smem);
#pragma unroll
    for (int r = 0; r < G; ++r) {
      float M = -INFINITY;
#pragma unroll
      for (int w = 0; w < kDecWarps; ++w) M = fmaxf(M, red_m[w][r]);
      float num = 0.f, den = 0.f;
#pragma unroll
      for (int w = 0; w < kDecWarps; ++w) {
        const float mw = red_m[w][r];
        const float wgt = (mw == -INFINITY) ? 0.f : exp2f((mw - M) * scale_log2);
        num += wgt * o_all[(w * 8 + r) * kHeadDim + dim];
        den += wgt * red_l[w][r];
      }
      out[static_cast<size_t>(b) * hq * kHeadDim + (kvh * G + r) * kHeadDim + dim] =
          __float2bfloat16_rn(num / den);
    }
  }
}

// ---------------------------------------------------------------------------
// Throughput variant: one WARP per (sequence, kv head).  When the batch offers at least a
// few (sequence, kv head) pairs per resident warp there is no reason to split one pair
// across warps: each warp streams its pair's pages through a private 3-stage ring and
// writes the normalised output itself — no cross-warp merge, no __syncthreads, and the
// page-table / Q-load / pipeline-fill latency is paid once per pair instead of once per
// two or three tiles.
// ---------------------------------------------------------------------------
template <int G>
__global__ void __launch_bounds__(kDecWarps * 32)
attn_decode_warp_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out,
                        const __nv_bfloat16* __restrict__ kv_layer,
                        const int32_t* __restrict__ page_table, int max_pages,
                        const int32_t* __restrict__ row_slot, const int32_t* __restrict__ ctx_len,
                        int n_pairs, int hq, int hkv, float scale_log2) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~static_cast<uintptr_t>(127));
  __shared__ uint64_t full_bar[kDecWarps][kDecStages];

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int pair = blockIdx.x * kDecWarps + warp;
  if (pair >= n_pairs) return;  // whole warp exits together; no block-wide barriers below
  const int b = pair / hkv;
  const int kvh = pair - b * hkv;
  const int slot = row_slot[b];
  const int L = ctx_len[b];
  const int n_tiles = (L + kPageTokens - 1) / kPageTokens;
  const int32_t* pt = page_table + static_cast<size_t>(slot) * max_pages;

  uint8_t* my_smem = smem + warp * kDecStages * kStageBytes;
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kDecStages; ++s) mbar_init(smem_u32(&full_bar[warp][s]), 1);
    fence_mbar_init();
  }
  __syncwarp();

  auto issue = [&](int tile, int stage) {
    const int page = pt[tile];
    const __nv_bfloat16* src =
        kv_layer + (static_cast<size_t>(page) * hkv + kvh) * (2 * kTileElems);
    const uint32_t bar = smem_u32(&full_bar[warp][stage]);
    mbar_arrive_expect_tx(bar, kStageBytes);
    bulk_load_1d(smem_u32(my_smem + stage * kStageBytes), src, kStageBytes, bar);
  };
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kDecStages; ++s)
      if (s < n_tiles) issue(s, s);
  }

  const int ldq = (hq + 2 * hkv) * kHeadDim;
  const int qr = lane >> 2;
  uint32_t qa[8][2];
  {
    const __nv_bfloat16* qp =
        qkv + static_cast<size_t>(b) * ldq + (kvh * G + qr) * kHeadDim + 2 * (lane & 3);
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
      if (qr < G) {
        qa[kk][0] = *reinterpret_cast<const uint32_t*>(qp + kk * 16);
        qa[kk][1] = *reinterpret_cast<const uint32_t*>(qp + kk * 16 + 8);
      } else {
        qa[kk][0] = 0u;
        qa[kk][1] = 0u;
      }
    }
  }

  float o[16][2];
#pragma unroll
  for (int i = 0; i < 16; ++i) o[i][0] = o[i][1] = 0.f;
  float m_run = -INFINITY, l_run = 0.f;
  const int lm = lane >> 3;
  const int lr = lane & 7;

  for (int tile = 0; tile < n_tiles; ++tile) {
    const int stage = tile % kDecStages;
    const uint32_t phase = (tile / kDecStages) & 1;
    mbar_wait(smem_u32(&full_bar[warp][stage]), phase);
    const uint32_t ks = smem_u32(my_smem + stage * kStageBytes);
    const uint32_t vs = ks + kTileBytes;
    float s0[4] = {0.f, 0.f, 0.f, 0.f};
    float s1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
      const int tok = (lm >> 1) * 8 + lr;
      const int chunk = kk * 2 + (lm & 1);
      uint32_t b0, b1, b2, b3;
      ldmatrix_x4(ks + tok * 256 + ((chunk ^ (tok & 7)) << 4), b0, b1, b2, b3);
      const uint32_t a[4] = {qa[kk][0], 0u, qa[kk][1], 0u};
      mma_bf16_16816(s0, a, b0, b1);
      mma_bf16_16816(s1, a, b2, b3);
    }
    const int tok0 = tile * kPageTokens + 2 * (lane & 3);
    float sv[4] = {s0[0], s0[1], s1[0], s1[1]};
    if (tok0 >= L) sv[0] = -INFINITY;
    if (tok0 + 1 >= L) sv[1] = -INFINITY;
    if (tok0 + 8 >= L) sv[2] = -INFINITY;
    if (tok0 + 9 >= L) sv[3] = -INFINITY;
    float mx = fmaxf(fmaxf(sv[0], sv[1]), fmaxf(sv[2], sv[3]));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    const float m_new = fmaxf(m_run, mx);
    const float alpha = exp2f((m_run - m_new) * scale_log2);
    float p[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) p[i] = exp2f((sv[i] - m_new) * scale_log2);
    float ps = p[0] + p[1] + p[2] + p[3];
    ps += __shfl_xor_sync(0xffffffffu, ps, 1);
    ps += __shfl_xor_sync(0xffffffffu, ps, 2);
    l_run = l_run * alpha + ps;
    m_run = m_new;
    const uint32_t pa[4] = {pack_bf16x2(p[0], p[1]), 0u, pack_bf16x2(p[2], p[3]), 0u};
#pragma unroll
    for (int nt = 0; nt < 16; nt += 2) {
      const int tok = (lm & 1) * 8 + lr;
      const int chunk = nt + (lm >> 1);
      uint32_t b0, b1, b2, b3;
      ldmatrix_x4_trans(vs + tok * 256 + ((chunk ^ (tok & 7)) << 4), b0, b1, b2, b3);
      float d0[4] = {o[nt][0] * alpha, o[nt][1] * alpha, 0.f, 0.f};
      float d1[4] = {o[nt + 1][0] * alpha, o[nt + 1][1] * alpha, 0.f, 0.f};
      mma_bf16_16816(d0, pa, b0, b1);
      mma_bf16_16816(d1, pa, b2, b3);
      o[nt][0] = d0[0];
      o[nt][1] = d0[1];
      o[nt + 1][0] = d1[0];
      o[nt + 1][1] = d1[1];
    }
    __syncwarp();
    const int next = tile + kDecStages;
    if (lane == 0 && next < n_tiles) {
      fence_proxy_async_smem();
      issue(next, stage);
    }
  }
  if (qr < G) {
    const float inv = 1.0f / l_run;
    __nv_bfloat16* op = out + static_cast<size_t>(b) * hq * kHeadDim + (kvh * G + qr) * kHeadDim +
                        2 * (lane & 3);
#pragma unroll
    for (int nt = 0; nt < 16; ++nt)
      *reinterpret_cast<__nv_bfloat162*>(op + nt * 8) =
          __floats2bfloat162_rn(o[nt][0] * inv, o[nt][1] * inv);
  }
}

template <int G>
int launch(const void* qkv, void* out, const void* kv_layer, const int32_t* page_table,
           int max_pages, const int32_t* row_slot, const int32_t* ctx_len, int B, int hq, int hkv,
           float scale, cudaStream_t stream) {
  auto kern = attn_decode_kernel<G>;
  SB_SET_MAX_SMEM(kern, kDecSmem);
  const int n_pairs = B * hkv;
  int sms = 0, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  // The warp-per-(sequence, kv head) kernel is the only one the engine uses: which kernel
  // runs must not depend on the batch size, or a row's greedy tokens would depend on its
  // neighbours (the two kernels merge partial softmaxes in different orders).  The 4-warp
  // split kernel stays for explicit requests (tests, latency experiments).
  (void)sms;
  if (!g_force_split || g_force_warp) {
    auto wk = attn_decode_warp_kernel<G>;
    SB_SET_MAX_SMEM(wk, kDecSmem);
    wk<<<(n_pairs + kDecWarps - 1) / kDecWarps, kDecWarps * 32, kDecSmem, stream>>>(
        static_cast<const __nv_bfloat16*>(qkv), static_cast<__nv_bfloat16*>(out),
        static_cast<const __nv_bfloat16*>(kv_layer), page_table, max_pages, row_slot, ctx_len,
        n_pairs, hq, hkv, scale * 1.4426950408889634f);
    SB_CUDA_CHECK(cudaGetLastError());
    return 0;
  }
  dim3 grid(hkv, B);
  kern<<<grid, kDecWarps * 32, kDecSmem, stream>>>(
      static_cast<const __nv_bfloat16*>(qkv), static_cast<__nv_bfloat16*>(out),
      static_cast<const __nv_bfloat16*>(kv_layer), page_table, max_pages, row_slot, ctx_len, hq,
      hkv, scale * 1.4426950408889634f);
  SB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

void attn_decode_force_variant(int v) {  // 0 auto, 1 split (4 warps per pair), 2 warp per pair
  g_force_split = v == 1;
  g_force_warp = v == 2;
}

int attn_decode(const void* qkv, void* out, const void* kv_layer, const int32_t* page_table,
                int max_pages, const int32_t* row_slot, const int32_t* ctx_len, int B, int hq,
                int hkv, float scale, cudaStream_t stream) {
  if (B <= 0) return 0;
  if (hkv <= 0 || hq % hkv != 0) {
    set_last_error("attn_decode: hq=%d not a multiple of hkv=%d", hq, hkv);
    return -1;
  }
  switch (hq / hkv) {
    case 1:
      return launch<1>(qkv, out, kv_layer, page_table, max_pages, row_slot, ctx_len, B, hq, hkv,
                       scale, stream);
    case 2:
      return launch<2>(qkv, out, kv_layer, page_table, max_pages, row_slot, ctx_len, B, hq, hkv,
                       scale, stream);
    case 4:
      return launch<4>(qkv, out, kv_layer, page_table, max_pages, row_slot, ctx_len, B, hq, hkv,
                       scale, stream);
    case 5:
      return launch<5>(qkv, out, kv_layer, page_table, max_pages, row_slot, ctx_len, B, hq, hkv,
                       scale, stream);
    case 8:
      return launch<8>(qkv, out, kv_layer, page_table, max_pages, row_slot, ctx_len, B, hq, hkv,
                       scale, stream);
    default:
      set_last_error("attn_decode: unsupported GQA group size %d", hq / hkv);
      return -1;
  }
}

}  // namespace sb
