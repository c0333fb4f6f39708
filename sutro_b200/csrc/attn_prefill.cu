// sutro_b200 — K3: causal prefill attention over the paged KV cache (varlen).
//
// The prompt's K/V have already been written to the cache by rope_kv_write, so
// new tokens attend to [cached prefix | themselves] through one code path; a
// shared system-prompt prefix is just a run of shared page ids.
//
// Work decomposition: CTA = (q tile, kv head) of one sequence.  The CTA has
// G query heads x ceil(QT/16) token sub-tiles warps, QT = 128/G (8 warps for
// G = 1, 2, 4, 8; 10 for G = 5, whose 25-token tile ends inside the second
// sub-tile), so all heads of a GQA group reuse each K/V page loaded into shared
// memory.  Pages stream
// through a 3-stage cp.async.bulk ring of 32-token super-tiles (two flat 8 KiB
// copies of pre-swizzled tiles per stage, see kernels.h) so that one barrier
// round and one softmax rescale cover 32 KV tokens; math is FlashAttention-2
// style on mma.sync m16n8k16 with fp32 online softmax.
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"

namespace sb {

namespace {

constexpr int kPfStages = 3;                    // ring of 32-token super-tiles (2 pages)
constexpr int kPfStageBytes = 4 * kTileBytes;   // K0 | V0 | K1 | V1
constexpr int kPfSmem = kPfStages * kPfStageBytes + 1024;
constexpr int kPfMaxPages = 1024;               // 16 k tokens of context per sequence

// warps per CTA: G heads x ceil(QT/16) sub-tiles
constexpr int pf_warps(int G) { return G * ((128 / G + 15) / 16); }

template <int G>
__global__ void __launch_bounds__(pf_warps(G) * 32, pf_warps(G) == 8 ? 2 : 1)
attn_prefill_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out,
                    const __nv_bfloat16* __restrict__ kv_layer,
                    const int32_t* __restrict__ page_table, int max_pages,
                    const int32_t* __restrict__ work, const int32_t* __restrict__ seq_slot,
                    const int32_t* __restrict__ seq_q_start, const int32_t* __restrict__ seq_q_len,
                    const int32_t* __restrict__ seq_past, int hq, int hkv, float scale_log2) {
  constexpr int QT = 128 / G;  // query tokens per CTA
  constexpr int kWarps = pf_warps(G);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~static_cast<uintptr_t>(127));
  __shared__ uint64_t full_bar[kPfStages];
  // page ids of this sequence, staged once: the producer lane must not sit on a dependent
  // global load (page table -> bulk copy) in every iteration while 7 warps wait at the barrier
  __shared__ int32_t s_pt[kPfMaxPages];

  const int seq = work[2 * blockIdx.x];
  const int qt0 = work[2 * blockIdx.x + 1];
  const int kvh = blockIdx.y;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int slot = seq_slot[seq];
  const int q_start = seq_q_start[seq];
  const int q_len = seq_q_len[seq];
  const int past = seq_past[seq];
  const int32_t* pt = page_table + static_cast<size_t>(slot) * max_pages;

  const int head = kvh * G + (warp % G);      // query head of this warp
  const int sub = warp / G;                   // 16-token sub-tile of this warp
  const int q0 = qt0 + sub * 16;              // first query token (within the sequence's new tokens)
  const int cta_q_end = min(qt0 + QT, q_len);  // exclusive
  // Tokens of this warp at or past q_end are not its to compute.  With QT a multiple of 16
  // no sub-tile crosses the tile's end, so that is the sequence's end; otherwise (G = 5) the
  // last sub-tile would also cover the first tokens of the next tile.
  const int q_end = QT % 16 == 0 ? q_len : cta_q_end;
  const int last_kv_pos = past + cta_q_end - 1;
  const int n_pages = last_kv_pos / kPageTokens + 1;
  const int n_super = (n_pages + 1) >> 1;      // 32-token super-tiles
  const int warp_last_pos = past + min(q0 + 16, q_end) - 1;  // causal horizon of this warp
  const bool warp_active = q0 < q_end;

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kPfStages; ++s) mbar_init(smem_u32(&full_bar[s]), 1);
    fence_mbar_init();
  }
  for (int i = threadIdx.x; i < n_pages; i += kWarps * 32) s_pt[i] = pt[i];
  __syncthreads();

  // one super-tile = up to two pages, each one flat 8 KiB copy (K tile + V tile)
  auto issue = [&](int sup, int stage) {
    const int p0 = 2 * sup;
    const bool two = p0 + 1 < n_pages;
    const uint32_t bar = smem_u32(&full_bar[stage]);
    const uint32_t dst = smem_u32(smem + stage * kPfStageBytes);
    mbar_arrive_expect_tx(bar, two ? 4 * kTileBytes : 2 * kTileBytes);
    bulk_load_1d(dst, kv_layer + (static_cast<size_t>(s_pt[p0]) * hkv + kvh) * (2 * kTileElems),
                 2 * kTileBytes, bar);
    if (two)
      bulk_load_1d(dst + 2 * kTileBytes,
                   kv_layer + (static_cast<size_t>(s_pt[p0 + 1]) * hkv + kvh) * (2 * kTileElems),
                   2 * kTileBytes, bar);
  };
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kPfStages - 1; ++s)
      if (s < n_super) issue(s, s);
  }

  // Q fragments for this warp's 16 tokens x 128 dims.
  const int ldq = (hq + 2 * hkv) * kHeadDim;
  const int r0 = lane >> 2;
  uint32_t qa[8][4];
  {
    const int t0 = q0 + r0, t1 = q0 + r0 + 8;
    const __nv_bfloat16* p0 =
        qkv + static_cast<size_t>(q_start + t0) * ldq + head * kHeadDim + 2 * (lane & 3);
    const __nv_bfloat16* p1 = p0 + static_cast<size_t>(8) * ldq;
    const bool v0 = t0 < q_end, v1 = t1 < q_end;
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
      qa[kk][0] = v0 ? *reinterpret_cast<const uint32_t*>(p0 + kk * 16) : 0u;
      qa[kk][1] = v1 ? *reinterpret_cast<const uint32_t*>(p1 + kk * 16) : 0u;
      qa[kk][2] = v0 ? *reinterpret_cast<const uint32_t*>(p0 + kk * 16 + 8) : 0u;
      qa[kk][3] = v1 ? *reinterpret_cast<const uint32_t*>(p1 + kk * 16 + 8) : 0u;
    }
  }

  float o[16][4];
#pragma unroll
  for (int i = 0; i < 16; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY};
  float l_run[2] = {0.f, 0.f};
  const int pos_r0 = past + q0 + r0;  // absolute position of row r0 (row r0+8: +8)

  const int lm = lane >> 3;
  const int lr = lane & 7;

  for (int sup = 0; sup < n_super; ++sup) {
    const int stage = sup % kPfStages;
    const uint32_t phase = (sup / kPfStages) & 1;
    // keep the ring full: the stage freed by the previous iteration's barrier
    if (threadIdx.x == 0) {
      const int nxt = sup + kPfStages - 1;
      if (nxt < n_super) {
        fence_proxy_async_smem();
        issue(nxt, nxt % kPfStages);
      }
    }
    mbar_wait(smem_u32(&full_bar[stage]), phase);

    if (warp_active && sup * 32 <= warp_last_pos) {
      const uint32_t base = smem_u32(smem + stage * kPfStageBytes);
      // second page of the super-tile: absent at an odd tail, or wholly above this warp's
      // causal horizon (then it is skipped: its shared memory may hold stale bytes)
      const bool two = (2 * sup + 1 < n_pages) && (sup * 32 + 16 <= warp_last_pos);
      float s[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i) s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f;
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const int tok = (lm >> 1) * 8 + lr;
        const int chunk = kk * 2 + (lm & 1);
        const uint32_t off = tok * 256 + ((chunk ^ (tok & 7)) << 4);
        uint32_t b0, b1, b2, b3;
        ldmatrix_x4(base + off, b0, b1, b2, b3);
        mma_bf16_16816(s[0], qa[kk], b0, b1);
        mma_bf16_16816(s[1], qa[kk], b2, b3);
        if (two) {
          ldmatrix_x4(base + 2 * kTileBytes + off, b0, b1, b2, b3);
          mma_bf16_16816(s[2], qa[kk], b0, b1);
          mma_bf16_16816(s[3], qa[kk], b2, b3);
        }
      }
      // causal mask (kv position > query position); a skipped second page counts as masked
      const int kp = sup * 32 + 2 * (lane & 3);
      float alpha[2];
      uint32_t pa[2][4];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int qp = pos_r0 + 8 * h;
        float sv[8];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const int k0 = kp + 8 * nt;
          const bool dead = (nt >= 2) && !two;
          sv[2 * nt] = (dead || k0 > qp) ? -INFINITY : s[nt][2 * h];
          sv[2 * nt + 1] = (dead || k0 + 1 > qp) ? -INFINITY : s[nt][2 * h + 1];
        }
        float mx = sv[0];
#pragma unroll
        for (int i = 1; i < 8; ++i) mx = fmaxf(mx, sv[i]);
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
        const float m_new = fmaxf(m_run[h], mx);
        // only padding rows can be fully masked here (position 0 is visible to every real row)
        const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
        alpha[h] = exp2f((m_run[h] - m_use) * scale_log2);
        float p[8], ps = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          p[i] = exp2f((sv[i] - m_use) * scale_log2);
          ps += p[i];
        }
        ps += __shfl_xor_sync(0xffffffffu, ps, 1);
        ps += __shfl_xor_sync(0xffffffffu, ps, 2);
        l_run[h] = l_run[h] * alpha[h] + ps;
        m_run[h] = m_new;
        pa[0][h] = pack_bf16x2(p[0], p[1]);
        pa[0][2 + h] = pack_bf16x2(p[2], p[3]);
        pa[1][h] = pack_bf16x2(p[4], p[5]);
        pa[1][2 + h] = pack_bf16x2(p[6], p[7]);
      }
#pragma unroll
      for (int nt = 0; nt < 16; nt += 2) {
        const int tok = (lm & 1) * 8 + lr;
        const int chunk = nt + (lm >> 1);
        const uint32_t off = kTileBytes + tok * 256 + ((chunk ^ (tok & 7)) << 4);
        o[nt][0] *= alpha[0];
        o[nt][1] *= alpha[0];
        o[nt][2] *= alpha[1];
        o[nt][3] *= alpha[1];
        o[nt + 1][0] *= alpha[0];
        o[nt + 1][1] *= alpha[0];
        o[nt + 1][2] *= alpha[1];
        o[nt + 1][3] *= alpha[1];
        uint32_t b0, b1, b2, b3;
        ldmatrix_x4_trans(base + off, b0, b1, b2, b3);
        mma_bf16_16816(o[nt], pa[0], b0, b1);
        mma_bf16_16816(o[nt + 1], pa[0], b2, b3);
        if (two) {
          ldmatrix_x4_trans(base + 2 * kTileBytes + off, b0, b1, b2, b3);
          mma_bf16_16816(o[nt], pa[1], b0, b1);
          mma_bf16_16816(o[nt + 1], pa[1], b2, b3);
        }
      }
    }
    __syncthreads();  // everyone is done with this stage -> it may be refilled
  }

  if (warp_active) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int t = q0 + r0 + 8 * h;
      if (t >= q_end) continue;
      const float inv = 1.0f / l_run[h];
      __nv_bfloat16* op = out + static_cast<size_t>(q_start + t) * hq * kHeadDim +
                          head * kHeadDim + 2 * (lane & 3);
#pragma unroll
      for (int nt = 0; nt < 16; ++nt) {
        *reinterpret_cast<__nv_bfloat162*>(op + nt * 8) =
            __floats2bfloat162_rn(o[nt][2 * h] * inv, o[nt][2 * h + 1] * inv);
      }
    }
  }
}

template <int G>
int launch(const void* qkv, void* out, const void* kv_layer, const int32_t* page_table,
           int max_pages, const int32_t* work, int n_work, const int32_t* seq_slot,
           const int32_t* seq_q_start, const int32_t* seq_q_len, const int32_t* seq_past, int hq,
           int hkv, float scale, cudaStream_t stream) {
  auto kern = attn_prefill_kernel<G>;
  SB_SET_MAX_SMEM(kern, kPfSmem);
  dim3 grid(n_work, hkv);
  kern<<<grid, pf_warps(G) * 32, kPfSmem, stream>>>(
      static_cast<const __nv_bfloat16*>(qkv), static_cast<__nv_bfloat16*>(out),
      static_cast<const __nv_bfloat16*>(kv_layer), page_table, max_pages, work, seq_slot,
      seq_q_start, seq_q_len, seq_past, hq, hkv, scale * 1.4426950408889634f);
  SB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

int attn_prefill_q_tile(int hq, int hkv) { return 128 / (hq / hkv); }

int attn_prefill(const void* qkv, void* out, const void* kv_layer, const int32_t* page_table,
                 int max_pages, const int32_t* work, int n_work, const int32_t* seq_slot,
                 const int32_t* seq_q_start, const int32_t* seq_q_len, const int32_t* seq_past,
                 int hq, int hkv, float scale, cudaStream_t stream) {
  if (n_work <= 0) return 0;
  if (hkv <= 0 || hq % hkv != 0) {
    set_last_error("attn_prefill: hq=%d not a multiple of hkv=%d", hq, hkv);
    return -1;
  }
  if (max_pages > kPfMaxPages) {
    set_last_error("attn_prefill: max_pages=%d exceeds the staged page-table size %d", max_pages,
                   kPfMaxPages);
    return -1;
  }
#define SB_PF(G)                                                                               \
  return launch<G>(qkv, out, kv_layer, page_table, max_pages, work, n_work, seq_slot,         \
                   seq_q_start, seq_q_len, seq_past, hq, hkv, scale, stream)
  switch (hq / hkv) {
    case 1: SB_PF(1);
    case 2: SB_PF(2);
    case 4: SB_PF(4);
    case 5: SB_PF(5);
    case 8: SB_PF(8);
    default:
      set_last_error("attn_prefill: unsupported GQA group size %d", hq / hkv);
      return -1;
  }
#undef SB_PF
}

}  // namespace sb
