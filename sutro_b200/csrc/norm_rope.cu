// sutro_b200 — K4/K5/K9: HBM-bound row kernels.
//   rmsnorm            one warp per row, 16-byte vector loads, warp-shuffle reduce
//   embed_gather       one warp per row copy
//   rope_kv_write      per-head q/k RMSNorm (Qwen3) + rotate-half RoPE, K/V scatter
//                      into the swizzled paged cache
//   l2_normalize_rows  embedding head (fp32 out)
// Rounding points follow the bf16 reference model (oracle/model_ref.py), which
// restates transformers 5.5.0 modeling_qwen3.py:50-66 (RMSNorm), :151-180 (RoPE),
// :248-264 (q/k norm before RoPE).
#include "common.cuh"
#include "kernels.h"

namespace sb {

namespace {

constexpr int kRowWarps = 4;

// NV = 16-byte vectors per lane held in registers (row length <= NV*32*8 elements): the row
// is read from HBM exactly once.  NV == 0 is the generic two-pass fallback for long rows.
template <int NV>
__global__ void __launch_bounds__(kRowWarps * 32)
rmsnorm_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ w,
               __nv_bfloat16* __restrict__ out, int rows, int d, float eps) {
  const int row = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const uint4* xr = reinterpret_cast<const uint4*>(x + static_cast<size_t>(row) * d);
  const uint4* wr = reinterpret_cast<const uint4*>(w);
  uint4* orow = reinterpret_cast<uint4*>(out + static_cast<size_t>(row) * d);
  const int nvec = d >> 3;
  float ss = 0.f;
  auto sq = [&](const uint4& v) {
    const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = unpack_bf16x2(u[j]);
      ss += f.x * f.x + f.y * f.y;
    }
  };
  auto emit = [&](int i, const uint4& v, float rstd) {
    const uint4 g = wr[i];
    const uint32_t u[4] = {v.x, v.y, v.z, v.w};
    const uint32_t gw[4] = {g.x, g.y, g.z, g.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = unpack_bf16x2(u[j]);
      const float2 wv = unpack_bf16x2(gw[j]);
      o[j] = pack_bf16x2(wv.x * bf16_round(f.x * rstd), wv.y * bf16_round(f.y * rstd));
    }
    orow[i] = make_uint4(o[0], o[1], o[2], o[3]);
  };
  if constexpr (NV > 0) {
    uint4 v[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int i = lane + 32 * k;
      v[k] = (i < nvec) ? ld_nc_v4(xr + i) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int k = 0; k < NV; ++k) sq(v[k]);
    ss = warp_sum(ss);
    const float rstd = rsqrtf(ss / static_cast<float>(d) + eps);
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int i = lane + 32 * k;
      if (i < nvec) emit(i, v[k], rstd);
    }
  } else {
    for (int i = lane; i < nvec; i += 32) sq(xr[i]);
    ss = warp_sum(ss);
    const float rstd = rsqrtf(ss / static_cast<float>(d) + eps);
    for (int i = lane; i < nvec; i += 32) emit(i, xr[i], rstd);  // second touch hits L1/L2
  }
}

__global__ void __launch_bounds__(kRowWarps * 32)
gather_rows_kernel(const int32_t* __restrict__ ids, const __nv_bfloat16* __restrict__ table,
                   __nv_bfloat16* __restrict__ out, int rows, int d) {
  const int row = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const uint4* src = reinterpret_cast<const uint4*>(table + static_cast<size_t>(ids[row]) * d);
  uint4* dst = reinterpret_cast<uint4*>(out + static_cast<size_t>(row) * d);
  for (int i = lane; i < (d >> 3); i += 32) dst[i] = src[i];
}

__global__ void __launch_bounds__(kRowWarps * 32)
l2norm_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ out, int rows, int d) {
  const int row = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const __nv_bfloat162* xr =
      reinterpret_cast<const __nv_bfloat162*>(x + static_cast<size_t>(row) * d);
  float ss = 0.f;
  for (int i = lane; i < (d >> 1); i += 32) {
    const float2 f = __bfloat1622float2(xr[i]);
    ss += f.x * f.x + f.y * f.y;
  }
  ss = warp_sum(ss);
  const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);
  float2* orow = reinterpret_cast<float2*>(out + static_cast<size_t>(row) * d);
  for (int i = lane; i < (d >> 1); i += 32) {
    const float2 f = __bfloat1622float2(xr[i]);
    orow[i] = make_float2(f.x * inv, f.y * inv);
  }
}

// One CTA per token; a half-warp per head (two heads per warp pass).  Lane l' = lane % 16
// owns dims {4l'..4l'+3} and {64+4l'..64+4l'+3}: the rotate-half partner of a dim lives in
// the same lane, loads/stores are 8 bytes wide, the per-head reduction is 4 shuffles.
constexpr int kRopeWarps = 8;

SB_DEVICE void unpack4(const uint2& u, float (&f)[4]) {
  const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
  f[0] = a.x, f[1] = a.y, f[2] = b.x, f[3] = b.y;
}
SB_DEVICE uint2 pack4(const float (&f)[4]) {
  return make_uint2(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]));
}

__global__ void __launch_bounds__(kRopeWarps * 32)
rope_kv_kernel(__nv_bfloat16* __restrict__ qkv, const __nv_bfloat16* __restrict__ q_norm_w,
               const __nv_bfloat16* __restrict__ k_norm_w, const __nv_bfloat16* __restrict__ cos_t,
               const __nv_bfloat16* __restrict__ sin_t, const int32_t* __restrict__ tok_slot,
               const int32_t* __restrict__ tok_pos, const int32_t* __restrict__ page_table,
               int max_pages, __nv_bfloat16* __restrict__ kv_layer, int hq, int hkv, float eps) {
  const int t = blockIdx.x;
  const int half = threadIdx.x >> 4;       // half-warp index within the CTA: 0..15
  const int l = threadIdx.x & 15;
  const int pos = tok_pos[t];
  const int slot = tok_slot[t];
  const int page = page_table[static_cast<size_t>(slot) * max_pages + pos / kPageTokens];
  const int r = pos % kPageTokens;
  const int nheads = hq + 2 * hkv;
  __nv_bfloat16* row = qkv + static_cast<size_t>(t) * nheads * kHeadDim;

  float cs[4], sn[4];  // cos/sin tables: [max_pos, 64] bf16, rounded like the reference
  unpack4(*reinterpret_cast<const uint2*>(cos_t + static_cast<size_t>(pos) * 64 + 4 * l), cs);
  unpack4(*reinterpret_cast<const uint2*>(sin_t + static_cast<size_t>(pos) * 64 + 4 * l), sn);

  // Every half-warp runs the same number of iterations (shuffles need full participation).
  // All of this thread's loads are issued before the first in-place store, so the memory
  // system sees up to 2*kMaxIt independent 8-byte requests per thread instead of a
  // load -> compute -> store chain per head.
  constexpr int kMaxIt = 4;  // supports up to 64 heads (q + k + v) per token
  const int iters = (nheads + 2 * kRopeWarps - 1) / (2 * kRopeWarps);
  uint2 rlo[kMaxIt], rhi[kMaxIt];
#pragma unroll
  for (int it = 0; it < kMaxIt; ++it) {
    const int h = it * 2 * kRopeWarps + half;
    if (it < iters && h < nheads) {
      rlo[it] = *reinterpret_cast<const uint2*>(row + h * kHeadDim + 4 * l);
      rhi[it] = *reinterpret_cast<const uint2*>(row + h * kHeadDim + 64 + 4 * l);
    } else {
      rlo[it] = rhi[it] = make_uint2(0u, 0u);
    }
  }
#pragma unroll
  for (int it = 0; it < kMaxIt; ++it) {
    if (it >= iters) break;
    const int h = it * 2 * kRopeWarps + half;
    const bool valid = h < nheads;
    const int hh = valid ? h : 0;
    __nv_bfloat16* hp = row + hh * kHeadDim;
    float lo[4], hi[4];
    unpack4(rlo[it], lo);
    unpack4(rhi[it], hi);
    const bool is_q = hh < hq;
    const bool is_k = !is_q && hh < hq + hkv;
    const __nv_bfloat16* nw = is_q ? q_norm_w : (is_k ? k_norm_w : nullptr);
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) ss += lo[i] * lo[i] + hi[i] * hi[i];
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);  // 16-lane sum
    if (nw != nullptr) {
      const float rstd = rsqrtf(ss / static_cast<float>(kHeadDim) + eps);
      float wl[4], wh[4];
      unpack4(*reinterpret_cast<const uint2*>(nw + 4 * l), wl);
      unpack4(*reinterpret_cast<const uint2*>(nw + 64 + 4 * l), wh);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        lo[i] = bf16_round(wl[i] * bf16_round(lo[i] * rstd));
        hi[i] = bf16_round(wh[i] * bf16_round(hi[i] * rstd));
      }
    }
    if (is_q || is_k) {
      // out[i] = x[i]*cos - x[i+64]*sin ; out[i+64] = x[i+64]*cos + x[i]*sin (bf16 op by op)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float a = bf16_round(lo[i] * cs[i]) + bf16_round(-hi[i] * sn[i]);
        const float b = bf16_round(hi[i] * cs[i]) + bf16_round(lo[i] * sn[i]);
        lo[i] = a;
        hi[i] = b;
      }
    }
    if (!valid) continue;
    const uint2 plo = pack4(lo), phi = pack4(hi);
    if (is_q) {
      *reinterpret_cast<uint2*>(hp + 4 * l) = plo;
      *reinterpret_cast<uint2*>(hp + 64 + 4 * l) = phi;
    } else {
      const int kvh = is_k ? (hh - hq) : (hh - hq - hkv);
      __nv_bfloat16* tile = kv_layer +
                            (static_cast<size_t>(page) * hkv + kvh) * (2 * kTileElems) +
                            (is_k ? 0 : kTileElems) + r * kHeadDim;
      const int c_lo = l >> 1;             // 16-byte chunk holding dims 4l..4l+3
      const int c_hi = c_lo + 8;
      const int within = (4 * l) & 7;      // 0 or 4 elements into the chunk
      *reinterpret_cast<uint2*>(tile + ((c_lo ^ (r & 7)) << 3) + within) = plo;
      *reinterpret_cast<uint2*>(tile + ((c_hi ^ (r & 7)) << 3) + within) = phi;
      if (is_k) {  // dense copy for the tcgen05 prefill attention (V is already in place)
        *reinterpret_cast<uint2*>(hp + 4 * l) = plo;
        *reinterpret_cast<uint2*>(hp + 64 + 4 * l) = phi;
      }
    }
  }
}

}  // namespace

int rmsnorm(const void* x, const void* w, void* out, int rows, int d, float eps,
            cudaStream_t stream) {
  if (rows <= 0) return 0;
  if (d % 8 != 0) {
    set_last_error("rmsnorm: d=%d must be a multiple of 8", d);
    return -1;
  }
  const int nvec = d >> 3;
  const dim3 grid((rows + kRowWarps - 1) / kRowWarps), block(kRowWarps * 32);
  auto* xp = static_cast<const __nv_bfloat16*>(x);
  auto* wp = static_cast<const __nv_bfloat16*>(w);
  auto* op = static_cast<__nv_bfloat16*>(out);
  if (x == out)  // in place: the streaming (non-coherent) loads must not be used
    rmsnorm_kernel<0><<<grid, block, 0, stream>>>(xp, wp, op, rows, d, eps);
  else if (nvec <= 32 * 4)
    rmsnorm_kernel<4><<<grid, block, 0, stream>>>(xp, wp, op, rows, d, eps);
  else if (nvec <= 32 * 10)
    rmsnorm_kernel<10><<<grid, block, 0, stream>>>(xp, wp, op, rows, d, eps);
  else if (nvec <= 32 * 16)
    rmsnorm_kernel<16><<<grid, block, 0, stream>>>(xp, wp, op, rows, d, eps);
  else if (nvec <= 32 * 20)  // d <= 5120 (Qwen3-14B / 32B)
    rmsnorm_kernel<20><<<grid, block, 0, stream>>>(xp, wp, op, rows, d, eps);
  else
    rmsnorm_kernel<0><<<grid, block, 0, stream>>>(xp, wp, op, rows, d, eps);
  SB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int embed_gather(const int32_t* ids, const void* table, void* out, int rows, int d,
                 cudaStream_t stream) {
  if (rows <= 0) return 0;
  if (d % 8 != 0) {
    set_last_error("embed_gather: d=%d must be a multiple of 8", d);
    return -1;
  }
  gather_rows_kernel<<<(rows + kRowWarps - 1) / kRowWarps, kRowWarps * 32, 0, stream>>>(
      ids, static_cast<const __nv_bfloat16*>(table), static_cast<__nv_bfloat16*>(out), rows, d);
  SB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int gather_rows(const int32_t* idx, const void* x, void* out, int rows, int d,
                cudaStream_t stream) {
  return embed_gather(idx, x, out, rows, d, stream);
}

int l2_normalize_rows(const void* x, float* out, int rows, int d, cudaStream_t stream) {
  if (rows <= 0) return 0;
  l2norm_kernel<<<(rows + kRowWarps - 1) / kRowWarps, kRowWarps * 32, 0, stream>>>(
      static_cast<const __nv_bfloat16*>(x), out, rows, d);
  SB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int rope_kv_write(void* qkv, const void* q_norm_w, const void* k_norm_w, const void* cos_tab,
                  const void* sin_tab, const int32_t* tok_slot, const int32_t* tok_pos,
                  const int32_t* page_table, int max_pages, void* kv_layer, int T, int hq,
                  int hkv, float eps, cudaStream_t stream) {
  if (T <= 0) return 0;
  if (hq + 2 * hkv > 64) {
    set_last_error("rope_kv_write: at most 64 heads (q+k+v) per token, got %d", hq + 2 * hkv);
    return -1;
  }
  rope_kv_kernel<<<T, kRopeWarps * 32, 0, stream>>>(
      static_cast<__nv_bfloat16*>(qkv), static_cast<const __nv_bfloat16*>(q_norm_w),
      static_cast<const __nv_bfloat16*>(k_norm_w), static_cast<const __nv_bfloat16*>(cos_tab),
      static_cast<const __nv_bfloat16*>(sin_tab), tok_slot, tok_pos, page_table, max_pages,
      static_cast<__nv_bfloat16*>(kv_layer), hq, hkv, eps);
  SB_CUDA_CHECK(cudaGetLastError());
  return 0;
}

}  // namespace sb
