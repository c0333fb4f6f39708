// sutro_b200 — K3 (tensor-core path): causal varlen prefill attention on tcgen05.
//
// The engine never splits a row's prompt over prefill steps, so a new token attends to
// [shared prefix | the row's own new tokens].  Both live in DENSE row-major buffers here:
// the fused QKV epilogue (gemm_tcgen05.cu) leaves post-norm / post-RoPE K and V in the qkv
// activation buffer next to q, and the shared prefix's K/V are kept per layer in a small
// dense side buffer.  Dense rows are what TMA wants: every operand tile below is one or a
// few cp.async.bulk.tensor boxes that land in shared memory already in the UMMA canonical
// 128-byte-swizzled layout.  (The paged cache is still written by the epilogue — decode reads
// it — and attn_prefill.cu remains the general paged-KV path for callers outside the engine.)
//
// Work item = (sequence, kv head, q tile).  A q tile packs QT = 128/G consecutive tokens x
// the G query heads of the kv head into the 128 rows of one UMMA M tile (row = token*G +
// head), so K/V are read once per GQA group and the causal frontier advances in QT-token
// steps.  For G = 5 (QT = 25) the tile fills 125 rows; rows 125..127 are padding: their Q
// rows are zero, their causal limit is the tile's last token and they never write output.
// KV is consumed in blocks of up to 128 tokens: first the prefix blocks, then the
// row's own blocks up to the tile's diagonal; the MMA N (and the PV K extent) is the valid
// token count rounded up to 16, so short sequences do not pay for padding.
//
// Persistent CTA, 224 threads, one per SM, software-pipelined across blocks AND items:
//   warps 4, 6  TMA producers Q tile (double-buffered) + K ring / V ring (2 stages each)
//   warp 5      MMA issuer    S = Q K^T -> TMEM S[2];  O (+)= P V -> TMEM O[2]
//   warps 0-3   softmax       thread == TMEM lane == tile row: tcgen05.ld S, running max with
//                             lazy rescale (threshold 2^8), exp2, P -> shared memory (bf16,
//                             K-major SW128), O rescale through tcgen05.ld/st when needed,
//                             epilogue O / l -> global
// Issue order of the MMA warp is S(g+1) before PV(g), so the tensor pipe computes the next
// block's scores while the softmax warps work on the current one.
//
// Results depend only on the sequence itself (block partition by absolute position, rescale
// decisions per row), never on which other sequences share the batch.
#include <algorithm>
#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "kernels.h"

namespace sb {

namespace {

constexpr int kTcThreads = 224;   // warps 0-3 softmax, 4 Q/K producer, 5 MMA issuer, 6 V producer
constexpr int kBlk = 128;                    // KV tokens per block (TMEM S columns)
constexpr int kHalfBytes = 128 * 128;        // [128 rows][64 bf16] = 16 KiB, one d-half / k-block
constexpr int kTileBytes2 = 2 * kHalfBytes;  // 32 KiB: Q tile, K block, V block, P block
constexpr int kBoxRows = 32;                 // K/V TMA box height
constexpr int kBoxBytes = kBoxRows * 128;    // 4 KiB
constexpr int kTcBarBytes = 256;
constexpr int kTcSmem = 7 * kTileBytes2 + kTcBarBytes + 1024;  // Q[2] K[2] V[2] P + barriers + align
constexpr float kRescaleThreshold = 8.0f;    // log2 units: P stays <= 2^8 before a forced rescale

// Q tile of a GQA group of G heads: QT = 128/G tokens x G heads, loaded as two d-halves of
// one TMA box {64, G, QT}.  The box (tc_maps) and the Q_FULL transaction count are both
// derived from here: a count that differs from the bytes TMA delivers never completes.
constexpr int tc_q_tokens(int G) { return 128 / G; }
constexpr int tc_q_rows(int G) { return tc_q_tokens(G) * G; }  // tile rows TMA fills
constexpr int tc_q_bytes(int G) { return 2 * tc_q_rows(G) * 64 * 2; }
template <int G>
constexpr bool tc_q_bytes_ok() {
  static_assert(tc_q_rows(G) <= 128 && tc_q_rows(G) > 120, "the q tile must nearly fill M = 128");
  static_assert(tc_q_bytes(G) == 2 * (kHalfBytes / 128) * tc_q_rows(G), "Q bytes != box bytes");
  static_assert(tc_q_bytes(G) % 16 == 0 && tc_q_bytes(G) <= kTileBytes2, "Q box overflows");
  static_assert(tc_q_rows(G) < 128 || tc_q_bytes(G) == kTileBytes2, "full tile != 32 KiB");
  return true;
}

struct TcGeom {
  int q_start, q_len, past, qt0, kvh;
  int n_pre, n_blocks;
};

template <int G>
SB_DEVICE TcGeom tc_geom(int item, int hkv, const int32_t* __restrict__ items,
                         const int32_t* __restrict__ seq_q_start,
                         const int32_t* __restrict__ seq_q_len,
                         const int32_t* __restrict__ seq_past) {
  constexpr int QT = 128 / G;
  TcGeom g;
  const int w = item / hkv;
  g.kvh = item - w * hkv;
  const int seq = items[2 * w];
  g.qt0 = items[2 * w + 1];
  g.q_start = seq_q_start[seq];
  g.q_len = seq_q_len[seq];
  g.past = seq_past[seq];
  g.n_pre = (g.past + kBlk - 1) / kBlk;
  const int own_end = min(g.q_len, g.qt0 + QT);  // exclusive causal frontier of the tile
  g.n_blocks = g.n_pre + (own_end + kBlk - 1) / kBlk;
  return g;
}

// block b of an item: source (prefix / own), first token, tokens the MMA covers (multiple of 16)
template <int G>
SB_DEVICE void tc_block(const TcGeom& g, int b, bool& is_pre, int& j0, int& n16) {
  constexpr int QT = 128 / G;
  is_pre = b < g.n_pre;
  int limit;
  if (is_pre) {
    j0 = b * kBlk;
    limit = g.past - j0;
  } else {
    j0 = (b - g.n_pre) * kBlk;
    limit = min(g.q_len, g.qt0 + QT) - j0;
  }
  limit = min(limit, kBlk);
  n16 = (limit + 15) & ~15;
}

#ifdef SB200_ATTN_TRACE
// Debug build only (tools/build_trace_lib.sh): CTA `g_tr_cta` stamps %clock at its pipeline
// hand-offs, kTrCap stamps per role, for `tools/attn_bench.py --trace`.  The pointer lives in
// the constant bank, so a stamp costs a compare, a CS2R and a store.  The product library is
// compiled without the macro and carries none of it.
constexpr int kTrCap = 1024;
__constant__ long long* g_tr = nullptr;
__constant__ int g_tr_cta = 0;
#define TR(role, idx)                                                                   \
  do {                                                                                  \
    if (g_tr != nullptr && static_cast<int>(blockIdx.x) == g_tr_cta && (idx) < kTrCap)  \
      g_tr[(role) * kTrCap + (idx)] = static_cast<long long>(clock());                 \
  } while (0)
#else
#define TR(role, idx) do { } while (0)
#endif

SB_DEVICE float ex2_approx(float x) {   // MUFU.EX2: 2^x, flushes denormals (x <= -126 -> 0)
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int G>
__global__ void __launch_bounds__(kTcThreads, 1)
attn_prefill_tc_kernel(const __grid_constant__ CUtensorMap tm_q,    // 3-D (d, head, token) over qkv
                       const __grid_constant__ CUtensorMap tm_kv,   // 2-D (col, token) over qkv
                       const __grid_constant__ CUtensorMap tm_pre,  // 3-D (col, token, layer)
                       __nv_bfloat16* __restrict__ out, const int32_t* __restrict__ items,
                       int n_items_total, const int32_t* __restrict__ seq_q_start,
                       const int32_t* __restrict__ seq_q_len, const int32_t* __restrict__ seq_past,
                       int hq, int hkv, int layer, float scale_log2) {
  constexpr int QT = 128 / G;
  constexpr int kQRows = tc_q_rows(G);
  constexpr bool kPad = kQRows < 128;  // G = 5: tile rows kQRows..127 are padding
  static_assert(QT == tc_q_tokens(G) && tc_q_bytes_ok<G>(), "q tile geometry");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(
      (reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  const uint32_t s_q = smem_u32(smem);                       // 2 x 32 KiB
  const uint32_t s_k = s_q + 2 * kTileBytes2;                // 2 x 32 KiB
  const uint32_t s_v = s_k + 2 * kTileBytes2;                // 2 x 32 KiB
  const uint32_t s_p = s_v + 2 * kTileBytes2;                // 32 KiB
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 7 * kTileBytes2);
  // barrier indices
  enum { Q_FULL = 0, Q_EMPTY = 2, K_FULL = 4, K_EMPTY = 6, V_FULL = 8, V_EMPTY = 10, S_FULL = 12,
         S_EMPTY = 14, P_FULL = 16, P_EMPTY = 17, O_FULL = 18, O_EMPTY = 20, N_BARS = 22 };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + N_BARS);
  auto bar = [&](int i) { return smem_u32(&bars[i]); };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tm_q);
    tma_prefetch_desc(&tm_kv);
    tma_prefetch_desc(&tm_pre);
  }
  if (warp == 5 && lane == 0) {
    for (int i = 0; i < N_BARS; ++i) {
      const bool from_softmax = (i >= S_EMPTY && i < S_EMPTY + 2) || i == P_FULL ||
                                (i >= O_EMPTY && i < O_EMPTY + 2);
      mbar_init(bar(i), from_softmax ? 4 : 1);  // softmax side: one arrival per warp
    }
    fence_mbar_init();
  }
  if (warp == 0) {
    tmem_alloc(smem_u32(tmem_slot), 512);
    tmem_relinquish();
  }
  if constexpr (kPad) {
    // TMA never writes the padding rows of the Q buffers: zero them once (both buffers, both
    // d-halves), so that their scores are exactly 0 and independent of what smem held before
    constexpr int kPadChunks = (128 - kQRows) * 128 / 16;  // 16-byte stores per d-half
    for (int i = threadIdx.x; i < 4 * kPadChunks; i += kTcThreads) {
      const int half = i / kPadChunks;  // (Q buffer, d-half) pair: 2 x 2
      const uint32_t a = s_q + half * kHalfBytes + kQRows * 128 + (i - half * kPadChunks) * 16;
      asm volatile("st.shared.v4.u32 [%0], {%1,%1,%1,%1};" ::"r"(a), "r"(0u) : "memory");
    }
    fence_proxy_async_smem();  // generic stores -> visible to the UMMA (async proxy)
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_s = tmem_base;        // S[sb] at columns sb*128
  const uint32_t tmem_o = tmem_base + 256;  // O[ob] at columns 256 + ob*128

  if (warp == 4 || warp == 6) {
    // ===================== TMA producers =====================
    // warp 4 streams Q tiles and K blocks, warp 6 the V blocks.  Two independent flows: a V
    // stage frees up only when its P.V has retired (after the softmax), a K stage as soon as
    // its S = Q.K^T has — one in-order producer would hold the next K block (and with it the
    // next S) hostage behind the wait for the previous block's V stage.
    const bool v_flow = warp == 6;
    if (lane == 0) {
      uint32_t g = 0;  // global block counter of this CTA
      uint32_t n = 0;  // item counter of this CTA
      for (int item = blockIdx.x; item < n_items_total; item += gridDim.x, ++n) {
        const TcGeom ge = tc_geom<G>(item, hkv, items, seq_q_start, seq_q_len, seq_past);
        if (!v_flow) {
          const uint32_t qb = n & 1;
          mbar_wait(bar(Q_EMPTY + qb), ((n >> 1) & 1) ^ 1);
          mbar_arrive_expect_tx(bar(Q_FULL + qb), tc_q_bytes(G));
          const uint32_t qd = s_q + qb * kTileBytes2;
          tma_load_3d(qd, &tm_q, bar(Q_FULL + qb), 0, ge.kvh * G, ge.q_start + ge.qt0);
          tma_load_3d(qd + kHalfBytes, &tm_q, bar(Q_FULL + qb), 64, ge.kvh * G,
                      ge.q_start + ge.qt0);
        }
        for (int b = 0; b < ge.n_blocks; ++b, ++g) {
          bool is_pre;
          int j0, n16;
          tc_block<G>(ge, b, is_pre, j0, n16);
          const int n32 = (n16 + kBoxRows - 1) / kBoxRows;
          const uint32_t st = g & 1, ph = ((g >> 1) & 1) ^ 1;
          const int kcol = is_pre ? ge.kvh * kHeadDim : (hq + ge.kvh) * kHeadDim;
          const int col = v_flow ? kcol + hkv * kHeadDim : kcol;
          const int row0 = is_pre ? j0 : ge.q_start + j0;
          const uint32_t full = bar((v_flow ? V_FULL : K_FULL) + st);
          const uint32_t base = (v_flow ? s_v : s_k) + st * kTileBytes2;
          mbar_wait(bar((v_flow ? V_EMPTY : K_EMPTY) + st), ph);
          TR(v_flow ? 1 : 0, 2 * g);
          mbar_arrive_expect_tx(full, n32 * 2 * kBoxBytes);
          for (int i = 0; i < n32; ++i) {
#pragma unroll
            for (int dh = 0; dh < 2; ++dh) {
              const uint32_t dst = base + dh * kHalfBytes + i * kBoxBytes;
              if (is_pre)
                tma_load_3d(dst, &tm_pre, full, col + dh * 64, row0 + i * kBoxRows, layer);
              else
                tma_load_2d(dst, &tm_kv, full, col + dh * 64, row0 + i * kBoxRows);
            }
          }
          TR(v_flow ? 1 : 0, 2 * g + 1);
        }
      }
    }
  } else if (warp == 5) {
    // ===================== MMA issuer =====================
    uint32_t g = 0, n = 0;
    bool have_pending = false;
    uint32_t p_g = 0, p_n16 = 0, p_ob = 0, p_opar = 0;
    bool p_first = false, p_last = false;

    auto do_pv = [&]() {
      if (lane == 0) TR(3, 4 * p_g);
      mbar_wait(bar(P_FULL), p_g & 1);
      if (lane == 0) TR(3, 4 * p_g + 1);
      mbar_wait(bar(V_FULL + (p_g & 1)), (p_g >> 1) & 1);
      if (lane == 0) TR(3, 4 * p_g + 2);
      if (p_first) mbar_wait(bar(O_EMPTY + p_ob), p_opar ^ 1);
      if (lane == 0) TR(3, 4 * p_g + 3);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t st = p_g & 1;
        const uint32_t d = tmem_o + p_ob * 128;
        const uint32_t idesc = umma_idesc_bf16(128, 128) | kUmmaBMajorMN;
        const int ksteps = static_cast<int>(p_n16) >> 4;
        for (int kk = 0; kk < ksteps; ++kk) {
          const uint64_t adesc = umma_desc_k_sw128(s_p + (kk >> 2) * kHalfBytes) + 2 * (kk & 3);
          const uint64_t bdesc =
              umma_desc_mn_sw128(s_v + st * kTileBytes2 + kk * 2048, kHalfBytes, 1024);
          tc_mma_f16(d, adesc, bdesc, idesc, (p_first && kk == 0) ? 0u : 1u);
        }
        tc_commit(bar(V_EMPTY + st));
        tc_commit(bar(P_EMPTY));
        if (p_last) tc_commit(bar(O_FULL + p_ob));
      }
      __syncwarp();
    };

    for (int item = blockIdx.x; item < n_items_total; item += gridDim.x, ++n) {
      const TcGeom ge = tc_geom<G>(item, hkv, items, seq_q_start, seq_q_len, seq_past);
      const uint32_t qb = n & 1;
      mbar_wait(bar(Q_FULL + qb), (n >> 1) & 1);
      for (int b = 0; b < ge.n_blocks; ++b, ++g) {
        bool is_pre;
        int j0, n16;
        tc_block<G>(ge, b, is_pre, j0, n16);
        const uint32_t st = g & 1;
        if (lane == 0) TR(2, 4 * g);
        if (b == 0 && lane == 0) TR(2, 4 * g + 3);
        mbar_wait(bar(K_FULL + st), (g >> 1) & 1);
        if (lane == 0) TR(2, 4 * g + 1);
        mbar_wait(bar(S_EMPTY + st), ((g >> 1) & 1) ^ 1);
        if (lane == 0) TR(2, 4 * g + 2);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t idesc = umma_idesc_bf16(128, n16);
          const uint32_t d = tmem_s + st * 128;
#pragma unroll
          for (int dh = 0; dh < 2; ++dh) {
            const uint64_t adesc = umma_desc_k_sw128(s_q + qb * kTileBytes2 + dh * kHalfBytes);
            const uint64_t bdesc = umma_desc_k_sw128(s_k + st * kTileBytes2 + dh * kHalfBytes);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              tc_mma_f16(d, adesc + 2 * k, bdesc + 2 * k, idesc, (dh | k) != 0 ? 1u : 0u);
          }
          tc_commit(bar(S_FULL + st));
          tc_commit(bar(K_EMPTY + st));
          if (b == ge.n_blocks - 1) tc_commit(bar(Q_EMPTY + qb));
        }
        __syncwarp();
        if (have_pending) do_pv();
        have_pending = true;
        p_g = g;
        p_n16 = static_cast<uint32_t>(n16);
        p_ob = n & 1;
        p_opar = (n >> 1) & 1;
        p_first = b == 0;
        p_last = b == ge.n_blocks - 1;
      }
    }
    if (have_pending) do_pv();
  } else {
    // ===================== softmax / correction / epilogue (warps 0-3) =====================
    const int r = warp * 32 + lane;       // tile row == TMEM lane
    const int t_in = r / G;               // token within the q tile
    const int h_in = r - t_in * G;        // query head within the GQA group
    // A padding row (kPad) takes the causal limit of the tile's last token: the largest in the
    // tile, so limits still grow with the lane (vmin below), and only columns that a real row
    // also reads.  It never writes output.
    const bool row_real = !kPad || r < kQRows;
    const int t_lim = kPad ? min(t_in, QT - 1) : t_in;
    const uint32_t lane_sel = static_cast<uint32_t>(warp * 32) << 16;
    const uint32_t p_row = s_p + r * 128;
    const int sw = r & 7;
    uint32_t g = 0, n = 0;
    float m_used = 0.f, l_run = 0.f;
    // The epilogue of an item is deferred until the first block of the NEXT item has been
    // handed to the tensor core: the wait for the last P.V (O_FULL) then overlaps useful work
    // instead of idling the softmax warps once per item (O is double-buffered).
    bool ep_pending = false;
    uint32_t ep_ob = 0, ep_par = 0;
    float ep_inv = 0.f;
    bool ep_row_ok = false;
    __nv_bfloat16* ep_dst = nullptr;
    auto flush_epilogue = [&]() {
      if (!ep_pending) return;
      ep_pending = false;
      mbar_wait(bar(O_FULL + ep_ob), ep_par);
      tc_fence_after();
      const uint32_t o_addr = tmem_o + ep_ob * 128 + lane_sel;
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {   // two 64-column halves: 64 live registers
        uint32_t v[2][32];
        tmem_ld_32x32(o_addr + half * 64, v[0]);
        tmem_ld_32x32(o_addr + half * 64 + 32, v[1]);
        tmem_ld_wait();
        if (half == 1) {  // the accumulator has left TMEM: hand O[ob] back before the stores
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar(O_EMPTY + ep_ob));
        }
        if (ep_row_ok) {
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint32_t o[16];
#pragma unroll
            for (int i = 0; i < 16; ++i)
              o[i] = pack_bf16x2(__uint_as_float(v[c][2 * i]) * ep_inv,
                                 __uint_as_float(v[c][2 * i + 1]) * ep_inv);
#pragma unroll
            for (int i = 0; i < 4; ++i)
              st_v4(ep_dst + half * 64 + c * 32 + 8 * i,
                    make_uint4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]));
          }
        }
      }
    };
    for (int item = blockIdx.x; item < n_items_total; item += gridDim.x, ++n) {
      const TcGeom ge = tc_geom<G>(item, hkv, items, seq_q_start, seq_q_len, seq_past);
      const int q_own = ge.qt0 + t_lim;   // index of this row's token among the own tokens
      const uint32_t ob = n & 1;
      for (int b = 0; b < ge.n_blocks; ++b, ++g) {
        bool is_pre;
        int j0, n16;
        tc_block<G>(ge, b, is_pre, j0, n16);
        // columns c of this block are valid for this row iff c < vlim
        const int vlim = min(is_pre ? ge.past - j0 : q_own - j0 + 1, n16);
        const uint32_t sb = g & 1;
        const int n_chunks = (n16 + 31) >> 5;
        if (threadIdx.x == 0) TR(4, 8 * g);
        mbar_wait(bar(S_FULL + sb), (g >> 1) & 1);
        if (threadIdx.x == 0) TR(4, 8 * g + 1);
        tc_fence_after();
        const uint32_t s_addr = tmem_s + sb * 128 + lane_sel;
        // ---- the whole score row into registers (one TMEM round trip), S[sb] released ----
        uint32_t v[4][32];
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c < n_chunks) tmem_ld_32x32(s_addr + c * 32, v[c]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(S_EMPTY + sb));
        if (threadIdx.x == 0) TR(4, 8 * g + 2);
        // One softmax warp per SM sub-partition: nothing hides ALU latency but ILP, and every
        // instruction counts.  So (a) chunks that are valid for every row of the warp (all but
        // the diagonal one: lane 0 holds the warp's smallest limit, limits grow with the lane)
        // take a path without per-element predicates, (b) max and sum run on four independent
        // accumulators, (c) exp2 is the bare MUFU (ex2.approx.ftz).
        const int vmin = __shfl_sync(0xffffffffu, vlim, 0);
        float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c < n_chunks) {
            if (c * 32 + 32 <= vmin) {
#pragma unroll
              for (int i = 0; i < 32; ++i) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(v[c][i]));
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (c * 32 + i < vlim) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(v[c][i]));
            }
          }
        float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
        mx *= scale_log2;  // scale > 0: max commutes with the scaling
        if (threadIdx.x == 0) TR(5, 4 * g);
        // ---- running max with lazy rescale ----
        float alpha = 1.f;
        bool need = false;
        if (b == 0) {
          m_used = (mx == -INFINITY) ? 0.f : mx;
          l_run = 0.f;
        } else if (mx > m_used + kRescaleThreshold) {
          alpha = ex2_approx(m_used - mx);
          m_used = mx;
          l_run *= alpha;
          need = true;
        }
        // ---- P = exp2(s*scale - m) -> bf16 (registers) ----
        float ps4[4] = {0.f, 0.f, 0.f, 0.f};
        const float neg_m = -m_used;
        if (threadIdx.x == 0) TR(5, 4 * g + 1);
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c < n_chunks) {
            if (c * 32 + 32 <= vmin) {
#pragma unroll
              for (int i = 0; i < 16; ++i) {   // packed pairs overwrite the scores in place
                const float p0 = ex2_approx(fmaf(__uint_as_float(v[c][2 * i]), scale_log2, neg_m));
                const float p1 =
                    ex2_approx(fmaf(__uint_as_float(v[c][2 * i + 1]), scale_log2, neg_m));
                ps4[i & 3] += p0 + p1;
                v[c][i] = pack_bf16x2(p0, p1);
              }
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const int c0 = c * 32 + 2 * i;
                float p0 = ex2_approx(fmaf(__uint_as_float(v[c][2 * i]), scale_log2, neg_m));
                float p1 = ex2_approx(fmaf(__uint_as_float(v[c][2 * i + 1]), scale_log2, neg_m));
                p0 = c0 < vlim ? p0 : 0.f;
                p1 = c0 + 1 < vlim ? p1 : 0.f;
                ps4[i & 3] += p0 + p1;
                v[c][i] = pack_bf16x2(p0, p1);
              }
            }
          }
        const float psum = (ps4[0] + ps4[1]) + (ps4[2] + ps4[3]);
        l_run += psum;
        // the previous block's PV must have retired before O is rescaled or P is overwritten
        if (threadIdx.x == 0) TR(4, 8 * g + 3);
        mbar_wait(bar(P_EMPTY), (g & 1) ^ 1);
        if (threadIdx.x == 0) TR(4, 8 * g + 4);
        if (__any_sync(0xffffffffu, need)) {
          tc_fence_after();
          const uint32_t o_addr = tmem_o + ob * 128 + lane_sel;
#pragma unroll 1
          for (int c = 0; c < 4; ++c) {
            uint32_t o[32];
            tmem_ld_32x32(o_addr + c * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st_32x32(o_addr + c * 32, o);
          }
          tmem_st_wait();
          tc_fence_before();
        }
        // ---- P -> shared memory (K-major, SW128): 32 columns = four 16-byte chunks ----
#pragma unroll
        for (int c = 0; c < 4; ++c)
          if (c < n_chunks) {
            const uint32_t base = p_row + (c >> 1) * kHalfBytes;
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              const int cc = (c & 1) * 4 + q4;
              asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(base + ((cc ^ sw) << 4)),
                           "r"(v[c][4 * q4]), "r"(v[c][4 * q4 + 1]), "r"(v[c][4 * q4 + 2]),
                           "r"(v[c][4 * q4 + 3])
                           : "memory");
            }
          }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(P_FULL));
        if (threadIdx.x == 0) TR(4, 8 * g + 5);
        flush_epilogue();
        if (threadIdx.x == 0) TR(4, 8 * g + 6);   // the previous item's, if any: the tensor core is busy with this block
        if (b == ge.n_blocks - 1) {
          ep_pending = true;
          ep_ob = ob;
          ep_par = (n >> 1) & 1;
          ep_inv = 1.0f / l_run;
          ep_row_ok = row_real && q_own < ge.q_len;
          ep_dst = out + static_cast<size_t>(ge.q_start + q_own) * (hq * kHeadDim) +
                   (ge.kvh * G + h_in) * kHeadDim;
        }
      }
    }
    flush_epilogue();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

struct TcMaps {
  CUtensorMap q, kv, pre;
};

struct TcKey {
  const void* qkv;
  const void* pre;
  int t_rows, hq, hkv, pre_rows, n_layers;
  bool operator==(const TcKey& o) const {
    return qkv == o.qkv && pre == o.pre && t_rows == o.t_rows && hq == o.hq && hkv == o.hkv &&
           pre_rows == o.pre_rows && n_layers == o.n_layers;
  }
};
struct TcKeyHash {
  size_t operator()(const TcKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.qkv) * 0x9E3779B97F4A7C15ull;
    h ^= reinterpret_cast<size_t>(k.pre) + (static_cast<size_t>(k.t_rows) << 7) +
         (static_cast<size_t>(k.pre_rows) << 29) + k.hq * 131 + k.hkv * 17 + k.n_layers;
    return h;
  }
};

int tc_maps(const TcKey& key, TcMaps* out) {
  static std::mutex mu;
  static std::unordered_map<TcKey, TcMaps, TcKeyHash> cache;
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) {
      *out = it->second;
      return 0;
    }
  }
  const int G = key.hq / key.hkv;
  const uint64_t ldq = static_cast<uint64_t>(key.hq + 2 * key.hkv) * kHeadDim;
  TcMaps m;
  {
    const uint64_t dims[3] = {static_cast<uint64_t>(kHeadDim), static_cast<uint64_t>(key.hq),
                              static_cast<uint64_t>(key.t_rows)};
    const uint64_t strides[2] = {kHeadDim * 2ull, ldq * 2ull};
    const uint32_t box[3] = {64u, static_cast<uint32_t>(G),
                             static_cast<uint32_t>(tc_q_tokens(G))};
    if (encode_tmap_bf16(&m.q, key.qkv, 3, dims, strides, box)) return -1;
  }
  {
    const uint64_t dims[2] = {ldq, static_cast<uint64_t>(key.t_rows)};
    const uint64_t strides[1] = {ldq * 2ull};
    const uint32_t box[2] = {64u, static_cast<uint32_t>(kBoxRows)};
    if (encode_tmap_bf16(&m.kv, key.qkv, 2, dims, strides, box)) return -1;
  }
  {
    // the prefix side buffer may be absent (no shared prefix): map the qkv buffer instead so
    // that the descriptor is valid; it is never dereferenced when every past == 0
    const bool have = key.pre != nullptr && key.pre_rows > 0;
    const uint64_t cols = 2ull * key.hkv * kHeadDim;
    const uint64_t rows = have ? key.pre_rows : 1;
    const uint64_t dims[3] = {have ? cols : 64ull, rows,
                              static_cast<uint64_t>(have ? key.n_layers : 1)};
    const uint64_t strides[2] = {(have ? cols : ldq) * 2ull, (have ? cols : ldq) * 2ull * rows};
    const uint32_t box[3] = {64u, static_cast<uint32_t>(kBoxRows), 1u};
    if (encode_tmap_bf16(&m.pre, have ? key.pre : key.qkv, 3, dims, strides, box)) return -1;
  }
  std::lock_guard<std::mutex> g(mu);
  cache.emplace(key, m);
  *out = m;
  return 0;
}

int tc_num_sms() {
  int dev = 0, n = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
  return n > 0 ? n : 148;
}

template <int G>
int launch_tc(const TcMaps& m, void* out, const int32_t* items, int n_items, const int32_t* qs,
              const int32_t* ql, const int32_t* past, int hq, int hkv, int layer, float scale,
              cudaStream_t stream) {
  auto kern = attn_prefill_tc_kernel<G>;
  SB_SET_MAX_SMEM(kern, kTcSmem);
  const int total = n_items * hkv;
  const int grid = std::min(total, tc_num_sms());
  kern<<<grid, kTcThreads, kTcSmem, stream>>>(m.q, m.kv, m.pre, static_cast<__nv_bfloat16*>(out),
                                              items, total, qs, ql, past, hq, hkv, layer,
                                              scale * 1.4426950408889634f);
  SB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace

int attn_prefill_dense(const void* qkv, int t_rows, void* out, const void* prefix_kv,
                       int prefix_rows, int n_layers, int layer, const int32_t* items, int n_items,
                       const int32_t* seq_q_start, const int32_t* seq_q_len,
                       const int32_t* seq_past, int hq, int hkv, float scale,
                       cudaStream_t stream) {
  if (n_items <= 0) return 0;
  if (hkv <= 0 || hq % hkv != 0) {
    set_last_error("attn_prefill_dense: hq=%d not a multiple of hkv=%d", hq, hkv);
    return -1;
  }
  if (layer < 0 || layer >= std::max(n_layers, 1)) {
    set_last_error("attn_prefill_dense: layer %d out of range", layer);
    return -1;
  }
  TcMaps m;
  if (tc_maps(TcKey{qkv, prefix_kv, t_rows, hq, hkv, prefix_rows, n_layers}, &m)) return -1;
#define SB_TC(G)                                                                             \
  return launch_tc<G>(m, out, items, n_items, seq_q_start, seq_q_len, seq_past, hq, hkv,    \
                      prefix_kv ? layer : 0, scale, stream)
  switch (hq / hkv) {
    case 1: SB_TC(1);
    case 2: SB_TC(2);
    case 4: SB_TC(4);
    case 5: SB_TC(5);
    case 8: SB_TC(8);
    default:
      set_last_error("attn_prefill_dense: unsupported GQA group size %d", hq / hkv);
      return -1;
  }
#undef SB_TC
}

}  // namespace sb

#ifdef SB200_ATTN_TRACE
extern "C" int sb200_attn_trace(long long* dev_buf, int cta) {
  if (cudaMemcpyToSymbol(sb::g_tr, &dev_buf, sizeof(dev_buf)) != cudaSuccess) return -1;
  if (cudaMemcpyToSymbol(sb::g_tr_cta, &cta, sizeof(cta)) != cudaSuccess) return -1;
  return 0;
}
#endif
