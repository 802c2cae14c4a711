// Bandwidth-bound kernels of the training step (reference: ForwardTransformer._train_step, model/models.py:464-482,
// losses utils/losses.py:41-70, Adam utils/training_config_manager.py:102-106): softmax forward/backward on materialised
// score rows, LayerNorm backward (with the fused bias / gamma / beta gradients), bias-gradient column sums, ReLU masks,
// loss + its gradient, length-regulator / embedding / head backward, fused Adam.
// All are coalesced row kernels; reductions across rows use shared-memory partials + fp32 atomics.
#include <cuda_fp16.h>
#include <algorithm>

#include "../../include/ttsb.h"
#include "ttsb_common.cuh"
#include "ttsb_host.h"

namespace ttsb {

__device__ __forceinline__ float wsum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float wmax(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ------------------------------------------------------------------------------------------------
// softmax over materialised score rows (training attention):  S fp32 (Z, T, ld) already scaled by 1/sqrt(dh)
// ------------------------------------------------------------------------------------------------
__global__ void softmax_fwd_kernel(const float* __restrict__ S, int Z, int H, int T, int Tk, int ld, const int* __restrict__ kv_len,
                                   float drop_p, uint32_t seed, uint32_t site, int flags, __nv_bfloat16* __restrict__ P_pre,
                                   __nv_bfloat16* __restrict__ P_drop) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= Z * T) return;
  const int lane = threadIdx.x & 31;
  const int z = row / T, t = row % T, b = z / H;
  int len = min(max(__ldg(kv_len + b), 0), Tk);
  const size_t base = (size_t)row * ld;
  // flags bit 1 (full queries): every query row is live (Aligner blocks); otherwise padded query rows are masked
  // downstream and written as zeros.  bit 0 (look-ahead mask): keys > t are masked.
  const bool live = (flags & 2) ? len > 0 : t < len;
  if (flags & 1) len = min(len, t + 1);
  float mx = -INFINITY;
  if (live)
    for (int k = lane; k < len; k += 32) mx = fmaxf(mx, S[base + k]);
  mx = wmax(mx);
  float sum = 0.f;
  if (live)
    for (int k = lane; k < len; k += 32) sum += __expf(S[base + k] - mx);
  sum = wsum(sum);
  const float inv = live ? 1.f / sum : 0.f;
  const uint32_t thresh = drop_p > 0.f ? (uint32_t)(drop_p * 4294967296.0) : 0u;
  const float keep_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  for (int k = lane; k < ld; k += 32) {
    float pv = (live && k < len) ? __expf(S[base + k] - mx) * inv : 0.f;
    P_pre[base + k] = __float2bfloat16_rn(pv);
    if (P_drop != P_pre) {
      const bool keep = drop_p <= 0.f || dropout_keep(seed, site, base + k, thresh);
      P_drop[base + k] = __float2bfloat16_rn(keep ? pv * keep_scale : 0.f);
    }
  }
}

// The same for rows of up to 1024 padded keys (every attention of the model at T <= 1024) with the row held in registers:
// ONE pass over S (16-byte loads, lane = 4 consecutive keys per 128-key group), exp evaluated once, 8-byte bf16 stores, one
// dropout hash per key pair.  NG = number of 128-key groups.
template <int NG>
__global__ void __launch_bounds__(256)
softmax_fwd_vec_kernel(const float* __restrict__ S, int Z, int H, int T, int Tk, int ld, const int* __restrict__ kv_len, float drop_p,
                       uint32_t seed, uint32_t site, int flags, __nv_bfloat16* __restrict__ P_pre, __nv_bfloat16* __restrict__ P_drop) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= Z * T) return;
  const int lane = threadIdx.x & 31;
  const int z = row / T, t = row % T, b = z / H;
  int len = min(max(__ldg(kv_len + b), 0), Tk);
  const size_t base = (size_t)row * ld;
  const bool live = (flags & 2) ? len > 0 : t < len;
  if (flags & 1) len = min(len, t + 1);
  if (!live) len = 0;
  float4 v[NG];
  float mx = -INFINITY;
#pragma unroll
  for (int i = 0; i < NG; ++i) {
    const int k = 4 * lane + 128 * i;
    v[i] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    if (k < len) {   // (ld is a multiple of 16, so a started group of four is inside the padded row)
      v[i] = __ldcs(reinterpret_cast<const float4*>(S + base + k));
      if (k + 1 >= len) v[i].y = -INFINITY;
      if (k + 2 >= len) v[i].z = -INFINITY;
      if (k + 3 >= len) v[i].w = -INFINITY;
      mx = fmaxf(mx, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w)));
    }
  }
  mx = wmax(mx);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NG; ++i) {
    v[i].x = __expf(v[i].x - mx); v[i].y = __expf(v[i].y - mx); v[i].z = __expf(v[i].z - mx); v[i].w = __expf(v[i].w - mx);
    sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  sum = wsum(sum);
  const float inv = len > 0 ? 1.f / sum : 0.f;
  const uint32_t thresh = dropout_thresh(drop_p);
  const float keep_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
#pragma unroll
  for (int i = 0; i < NG; ++i) {
    const int k = 4 * lane + 128 * i;
    if (k < ld) {
      float pv[4] = {v[i].x * inv, v[i].y * inv, v[i].z * inv, v[i].w * inv};
      if (len == 0) pv[0] = pv[1] = pv[2] = pv[3] = 0.f;     // exp(-inf - (-inf)) is NaN on dead rows
      const __nv_bfloat162 a = __floats2bfloat162_rn(pv[0], pv[1]), c = __floats2bfloat162_rn(pv[2], pv[3]);
      uint2 pk;
      pk.x = *reinterpret_cast<const uint32_t*>(&a);
      pk.y = *reinterpret_cast<const uint32_t*>(&c);
      *reinterpret_cast<uint2*>(P_pre + base + k) = pk;
      if (P_drop != P_pre) {
        bool k0 = true, k1 = true, k2 = true, k3 = true;
        if (drop_p > 0.f) {
          dropout_keep2(seed, site, base + k, thresh, k0, k1);
          dropout_keep2(seed, site, base + k + 2, thresh, k2, k3);
        }
        const __nv_bfloat162 d0 = __floats2bfloat162_rn(k0 ? pv[0] * keep_scale : 0.f, k1 ? pv[1] * keep_scale : 0.f);
        const __nv_bfloat162 d1 = __floats2bfloat162_rn(k2 ? pv[2] * keep_scale : 0.f, k3 ? pv[3] * keep_scale : 0.f);
        pk.x = *reinterpret_cast<const uint32_t*>(&d0);
        pk.y = *reinterpret_cast<const uint32_t*>(&d1);
        *reinterpret_cast<uint2*>(P_drop + base + k) = pk;
      }
    }
  }
}

// dS = scale * P_pre * (dPp - sum_k P_pre dPp),  dPp = dP * keep/(1-p).  Two light passes over the row (the second one
// hits L2); keeping the row in registers instead was measured 2-4x slower (occupancy).
__global__ void softmax_bwd_kernel(const __nv_bfloat16* __restrict__ P_pre, const float* __restrict__ dP, int Z, int H, int T, int Tk,
                                   int ld, const int* __restrict__ kv_len, float scale, float drop_p, uint32_t seed, uint32_t site,
                                   int flags, __nv_bfloat16* __restrict__ dS) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= Z * T) return;
  const int lane = threadIdx.x & 31;
  const int z = row / T, t = row % T, b = z / H;
  int len = min(max(__ldg(kv_len + b), 0), Tk);
  const size_t base = (size_t)row * ld;
  const bool live = (flags & 2) ? len > 0 : t < len;
  if (flags & 1) len = min(len, t + 1);
  const uint32_t thresh = dropout_thresh(drop_p);
  const float keep_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  float dot = 0.f;
  if (live)
    for (int k = lane; k < len; k += 32) {
      const bool keep = drop_p <= 0.f || dropout_keep(seed, site, base + k, thresh);
      const float g = keep ? dP[base + k] * keep_scale : 0.f;
      dot += __bfloat162float(P_pre[base + k]) * g;
    }
  dot = wsum(dot);
  for (int k = lane; k < ld; k += 32) {
    float v = 0.f;
    if (live && k < len) {
      const bool keep = drop_p <= 0.f || dropout_keep(seed, site, base + k, thresh);
      const float g = keep ? dP[base + k] * keep_scale : 0.f;
      v = scale * __bfloat162float(P_pre[base + k]) * (g - dot);
    }
    dS[base + k] = __float2bfloat16_rn(v);
  }
}

// ------------------------------------------------------------------------------------------------
// LayerNorm backward (Keras non-fused forward: y = (u-mean)*rsqrt(var+eps)*gamma + beta), one warp per row.
//   dz fp32 (M, ld), u fp32 (M, ld) pre-LN values, C valid columns.  Rows t >= row_len[b] carry zero gradient.
//   outputs: du fp32 (optional), g bf16 = du (* relu mask u>0 if relu_mask) (* dropout mask) for the GEMMs,
//   dgamma/dbeta accumulated with atomics.  dz_drop_*: dropout applied AFTER the LayerNorm in the forward pass.
// ------------------------------------------------------------------------------------------------
template <int MAXV>
__global__ void layernorm_bwd_kernel(const float* __restrict__ dz, const float* __restrict__ u, const float* __restrict__ gamma,
                                     int M, int T, int C, int ld, float eps, const int* __restrict__ row_len, int relu_mask,
                                     float pre_drop_p, uint32_t pre_site, float post_drop_p, uint32_t post_site, uint32_t seed,
                                     float* __restrict__ du, __nv_bfloat16* __restrict__ g_out, float* __restrict__ dgamma,
                                     float* __restrict__ dbeta, float* __restrict__ dbias) {
  extern __shared__ float part[];  // [3][C] per block: dgamma, dbeta, dbias partials
  for (int c = threadIdx.x; c < 3 * C; c += blockDim.x) part[c] = 0.f;
  __syncthreads();
  const int warps = blockDim.x >> 5, lane = threadIdx.x & 31;
  constexpr int RPW = 4;  // rows per warp; column partials stay in registers across them (MAXV = ceil(C/32))
  float acc_g[MAXV], acc_b[MAXV], acc_x[MAXV];
#pragma unroll
  for (int i = 0; i < MAXV; ++i) acc_g[i] = acc_b[i] = acc_x[i] = 0.f;
  const uint32_t post_thresh = dropout_thresh(post_drop_p);
  const float post_scale = post_drop_p > 0.f ? 1.f / (1.f - post_drop_p) : 1.f;
  const uint32_t pre_thresh = dropout_thresh(pre_drop_p);
  const float pre_scale = pre_drop_p > 0.f ? 1.f / (1.f - pre_drop_p) : 1.f;
  for (int rr = 0; rr < RPW; ++rr) {
    const int row = (blockIdx.x * warps + (threadIdx.x >> 5)) * RPW + rr;
    if (row >= M) break;
    const int b = row / T, t = row % T;
    const bool live = row_len == nullptr || t < __ldg(row_len + b);
    const size_t base = (size_t)row * ld;
    float uv[MAXV], gz[MAXV];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      uv[i] = (c < C) ? u[base + c] : 0.f;
      float g = (c < C && live) ? dz[base + c] : 0.f;
      if (post_drop_p > 0.f && c < C) g = dropout_keep(seed, post_site, base + c, post_thresh) ? g * post_scale : 0.f;
      gz[i] = g;
      s += uv[i];
    }
    const float mean = wsum(s) / C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      const float d = (c < C) ? uv[i] - mean : 0.f;
      q += d * d;
    }
    const float rstd = rsqrtf(wsum(q) / C + eps);
    float sg = 0.f, sgx = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < C) {
        const float xh = (uv[i] - mean) * rstd;
        const float gg = gz[i] * __ldg(gamma + c);
        sg += gg;
        sgx += gg * xh;
        acc_g[i] += gz[i] * xh;
        acc_b[i] += gz[i];
      }
    }
    sg = wsum(sg) / C;
    sgx = wsum(sgx) / C;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < ld) {
        float d = 0.f;
        if (c < C) {
          const float xh = (uv[i] - mean) * rstd;
          d = rstd * (gz[i] * __ldg(gamma + c) - sg - xh * sgx);
        }
        if (du) du[base + c] = d;
        float gv = d;
        if (relu_mask && !(uv[i] > 0.f)) gv = 0.f;
        if (pre_drop_p > 0.f) gv = dropout_keep(seed, pre_site, base + c, pre_thresh) ? gv * pre_scale : 0.f;
        if (g_out) g_out[base + c] = __float2bfloat16_rn(gv);
        if (c < C) acc_x[i] += gv;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int c = lane + 32 * i;
    if (c < C) {
      atomicAdd(part + c, acc_g[i]);
      atomicAdd(part + C + c, acc_b[i]);
      atomicAdd(part + 2 * C + c, acc_x[i]);
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    atomicAdd(dgamma + c, part[c]);
    atomicAdd(dbeta + c, part[C + c]);
    if (dbias) atomicAdd(dbias + c, part[2 * C + c]);
  }
}

// Same contract for rows whose width fills whole 128-column groups (C == ld, C % 128 == 0: every block LayerNorm of the
// model): a lane owns 4 consecutive columns per group (16-byte loads / stores, 8-byte bf16 stores), warps walk the rows with
// a grid stride and fetch row r+1 while the shuffle reductions of row r are in flight, and the column partials
// (dgamma, dbeta, dbias) stay in registers for the whole kernel: one shared-memory reduction and C*3 global atomics per block
// instead of per 32 rows.
template <int NG>
__global__ void __launch_bounds__(256)
layernorm_bwd_vec_kernel(const float* __restrict__ dz, const float* __restrict__ u, const float* __restrict__ gamma, int M, int T,
                         float eps, const int* __restrict__ row_len, int relu_mask, float pre_drop_p, uint32_t pre_site,
                         float post_drop_p, uint32_t post_site, uint32_t seed, float* __restrict__ du,
                         __nv_bfloat16* __restrict__ g_out, float* __restrict__ dgamma, float* __restrict__ dbeta,
                         float* __restrict__ dbias) {
  constexpr int C = NG * 128;
  __shared__ float part[3 * C];
  for (int c = threadIdx.x; c < 3 * C; c += blockDim.x) part[c] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int wid = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  const uint32_t post_thresh = dropout_thresh(post_drop_p), pre_thresh = dropout_thresh(pre_drop_p);
  const float post_scale = post_drop_p > 0.f ? 1.f / (1.f - post_drop_p) : 1.f;
  const float pre_scale = pre_drop_p > 0.f ? 1.f / (1.f - pre_drop_p) : 1.f;
  float4 gam[NG], acc_g[NG], acc_b[NG], acc_x[NG];
#pragma unroll
  for (int i = 0; i < NG; ++i) {
    gam[i] = __ldg(reinterpret_cast<const float4*>(gamma + 4 * lane + 128 * i));
    acc_g[i] = acc_b[i] = acc_x[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  // mask hash of element pair k of a row: mix((xrow + k*C1) ^ hterm); the host routes tensors of >= 2^33 elements to the
  // scalar kernel, so the pair index fits 32 bits (no 64-bit index arithmetic per pair)
  const uint32_t hterm_post = dropout_hterm(seed, post_site, 0u), hterm_pre = dropout_hterm(seed, pre_site, 0u);
  const uint32_t post_t16 = post_thresh >> 16, pre_t16 = pre_thresh >> 16;
  float4 un[NG], gn[NG];
  auto fetch = [&](int row) {
    const size_t base = (size_t)row * C;
#pragma unroll
    for (int i = 0; i < NG; ++i) {
      un[i] = __ldcs(reinterpret_cast<const float4*>(u + base + 4 * lane + 128 * i));
      gn[i] = __ldcs(reinterpret_cast<const float4*>(dz + base + 4 * lane + 128 * i));
    }
  };
  int row = wid;
  if (row < M) fetch(row);
  for (; row < M; row += nwarps) {
    float4 uv[NG], gz[NG];
#pragma unroll
    for (int i = 0; i < NG; ++i) { uv[i] = un[i]; gz[i] = gn[i]; }
    if (row + nwarps < M) fetch(row + nwarps);
    const int b = row / T, t = row % T;
    const bool live = row_len == nullptr || t < __ldg(row_len + b);
    const size_t base = (size_t)row * C;
    const uint32_t xl = ((uint32_t)(base >> 1) + 2u * lane) * DROPOUT_C1;   // pair of elements 4*lane, 4*lane+1 of the row
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NG; ++i) {
      float* g4 = reinterpret_cast<float*>(&gz[i]);
      bool kk[4] = {true, true, true, true};
      if (post_drop_p > 0.f) {
        const uint32_t h0 = dropout_mix((xl + (uint32_t)(64 * i) * DROPOUT_C1) ^ hterm_post);
        const uint32_t h1 = dropout_mix((xl + (uint32_t)(64 * i + 1) * DROPOUT_C1) ^ hterm_post);
        kk[0] = (h0 & 0xffffu) >= post_t16; kk[1] = (h0 >> 16) >= post_t16;
        kk[2] = (h1 & 0xffffu) >= post_t16; kk[3] = (h1 >> 16) >= post_t16;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) g4[j] = (live && kk[j]) ? g4[j] * post_scale : 0.f;
      s += (uv[i].x + uv[i].y) + (uv[i].z + uv[i].w);
    }
    const float mean = wsum(s) * (1.f / C);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NG; ++i) {
      const float a = uv[i].x - mean, b2 = uv[i].y - mean, c2 = uv[i].z - mean, d2 = uv[i].w - mean;
      q += (a * a + b2 * b2) + (c2 * c2 + d2 * d2);
    }
    const float rstd = rsqrtf(wsum(q) * (1.f / C) + eps);
    float sg = 0.f, sgx = 0.f;
#pragma unroll
    for (int i = 0; i < NG; ++i) {
      const float* u4 = reinterpret_cast<const float*>(&uv[i]);
      const float* g4 = reinterpret_cast<const float*>(&gz[i]);
      const float* m4 = reinterpret_cast<const float*>(&gam[i]);
      float* ag = reinterpret_cast<float*>(&acc_g[i]);
      float* ab = reinterpret_cast<float*>(&acc_b[i]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float xh = (u4[j] - mean) * rstd;
        const float gg = g4[j] * m4[j];
        sg += gg;
        sgx = fmaf(gg, xh, sgx);
        ag[j] = fmaf(g4[j], xh, ag[j]);
        ab[j] += g4[j];
      }
    }
    // two reductions in one pass over the shuffle network
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      sg += __shfl_xor_sync(0xffffffffu, sg, o);
      sgx += __shfl_xor_sync(0xffffffffu, sgx, o);
    }
    sg *= (1.f / C);
    sgx *= (1.f / C);
#pragma unroll
    for (int i = 0; i < NG; ++i) {
      const float* u4 = reinterpret_cast<const float*>(&uv[i]);
      const float* g4 = reinterpret_cast<const float*>(&gz[i]);
      const float* m4 = reinterpret_cast<const float*>(&gam[i]);
      float* ax = reinterpret_cast<float*>(&acc_x[i]);
      float d4[4], gv[4];
      bool kp[4] = {true, true, true, true};
      if (pre_drop_p > 0.f) {
        const uint32_t h0 = dropout_mix((xl + (uint32_t)(64 * i) * DROPOUT_C1) ^ hterm_pre);
        const uint32_t h1 = dropout_mix((xl + (uint32_t)(64 * i + 1) * DROPOUT_C1) ^ hterm_pre);
        kp[0] = (h0 & 0xffffu) >= pre_t16; kp[1] = (h0 >> 16) >= pre_t16;
        kp[2] = (h1 & 0xffffu) >= pre_t16; kp[3] = (h1 >> 16) >= pre_t16;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float xh = (u4[j] - mean) * rstd;
        d4[j] = rstd * (g4[j] * m4[j] - sg - xh * sgx);
        float v = d4[j];
        if (relu_mask && !(u4[j] > 0.f)) v = 0.f;
        v = kp[j] ? v * pre_scale : 0.f;
        gv[j] = v;
        ax[j] += v;
      }
      const size_t o = base + 4 * lane + 128 * i;
      if (du) __stcs(reinterpret_cast<float4*>(du + o), make_float4(d4[0], d4[1], d4[2], d4[3]));
      if (g_out) {
        const __nv_bfloat162 lo = __floats2bfloat162_rn(gv[0], gv[1]), hi = __floats2bfloat162_rn(gv[2], gv[3]);
        uint2 pk;
        pk.x = *reinterpret_cast<const uint32_t*>(&lo);
        pk.y = *reinterpret_cast<const uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(g_out + o) = pk;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < NG; ++i) {
    const float* ag = reinterpret_cast<const float*>(&acc_g[i]);
    const float* ab = reinterpret_cast<const float*>(&acc_b[i]);
    const float* ax = reinterpret_cast<const float*>(&acc_x[i]);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = 4 * lane + 128 * i + j;
      atomicAdd(part + c, ag[j]);
      atomicAdd(part + C + c, ab[j]);
      atomicAdd(part + 2 * C + c, ax[j]);
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    atomicAdd(dgamma + c, part[c]);
    atomicAdd(dbeta + c, part[C + c]);
    if (dbias) atomicAdd(dbias + c, part[2 * C + c]);
  }
}

// column sums of a bf16 matrix (rows, ld)[:, :C] -> fp32 [C] (accumulated): bias gradients.
// Block = 8 warps x 128 rows; a warp reads 512 contiguous bytes of a row (32 lanes x 8 bf16), partials meet in smem.
// Columns [k*seg, (k+1)*seg) go to out_k (k = 0..2; seg >= C: a single output): the q/k/v bias gradients are three
// separate parameters but one (rows, 3d) gradient buffer.
__global__ void colsum_bf16_kernel(const __nv_bfloat16* __restrict__ x, int64_t rows, int C, int ld, float* __restrict__ out,
                                   int seg, float* __restrict__ out1, float* __restrict__ out2) {
  __shared__ float red[8][256];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c0 = blockIdx.x * 256 + lane * 8;
  const int64_t r0 = (int64_t)blockIdx.y * 128;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (c0 < C) {
    for (int64_t r = r0 + w; r < r0 + 128 && r < rows; r += 8) {
      const uint4 v = *reinterpret_cast<const uint4*>(x + r * ld + c0);
      const __nv_bfloat16* h = reinterpret_cast<const __nv_bfloat16*>(&v);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += __bfloat162float(h[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[w][lane * 8 + j] = acc[j];
  __syncthreads();
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c < C) {
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) sum += red[k][threadIdx.x];
    const int k = c / seg;
    atomicAdd((k == 0 ? out : (k == 1 ? out1 : out2)) + (c - k * seg), sum);
  }
}

// dy (bf16, in place) *= (h > 0)
__global__ void relu_bwd_kernel(__nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ h, int64_t n) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (i >= n) return;
  uint4 g = *reinterpret_cast<const uint4*>(dy + i);
  const uint4 hv = *reinterpret_cast<const uint4*>(h + i);
  __nv_bfloat16* gp = reinterpret_cast<__nv_bfloat16*>(&g);
  const __nv_bfloat16* hp = reinterpret_cast<const __nv_bfloat16*>(&hv);
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (!(__bfloat162float(hp[j]) > 0.f)) gp[j] = __float2bfloat16(0.f);
  *reinterpret_cast<uint4*>(dy + i) = g;
}

// The same with the bias gradient of the layer that produced h: colsum[c] += sum over rows of the masked dy (C == ld).
// Block = 8 warps x 128 rows x 256 columns, like colsum_bf16_kernel: one pass over dy / h instead of two.
__global__ void relu_bwd_colsum_kernel(__nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ h, int64_t rows, int C,
                                       float* __restrict__ colsum) {
  __shared__ float red[8][256];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c0 = blockIdx.x * 256 + lane * 8;
  const int64_t r0 = (int64_t)blockIdx.y * 128;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (c0 < C) {
    for (int64_t r = r0 + w; r < r0 + 128 && r < rows; r += 8) {
      uint4 g = *reinterpret_cast<const uint4*>(dy + r * C + c0);
      const uint4 hv = *reinterpret_cast<const uint4*>(h + r * C + c0);
      __nv_bfloat16* gp = reinterpret_cast<__nv_bfloat16*>(&g);
      const __nv_bfloat16* hp = reinterpret_cast<const __nv_bfloat16*>(&hv);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (!(__bfloat162float(hp[j]) > 0.f)) gp[j] = __float2bfloat16(0.f);
        acc[j] += __bfloat162float(gp[j]);
      }
      *reinterpret_cast<uint4*>(dy + r * C + c0) = g;
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[w][lane * 8 + j] = acc[j];
  __syncthreads();
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c < C) {
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) sum += red[k][threadIdx.x];
    atomicAdd(colsum + c, sum);
  }
}

// fp32 (rows, C) -> bf16 (rows, ld_out >= C), zero in the padding columns (K of a GEMM must be a multiple of 64)
__global__ void cast_bf16_pad_kernel(const float* __restrict__ x, int64_t rows, int C, __nv_bfloat16* __restrict__ out, int ld_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * ld_out) return;
  const int c = (int)(i % ld_out);
  const int64_t r = i / ld_out;
  out[i] = __float2bfloat16_rn(c < C ? x[r * C + c] : 0.f);
}

// ------------------------------------------------------------------------------------------------
// mean absolute error over ALL elements (utils/losses.py:41-49 with mask=None) and its gradient
//   pred (rows, ld_pred)[:, :C] vs target (rows_t, C): rows beyond rows_valid get zero gradient
// ------------------------------------------------------------------------------------------------
__global__ void mae_loss_kernel(const float* __restrict__ pred, int64_t B, int64_t Tp, int64_t Tt, int C, const float* __restrict__ tgt_f,
                                const int* __restrict__ tgt_i, float weight, float* __restrict__ loss_out, float* __restrict__ grad) {
  // pred (B, Tp, C), target (B, Tt, C) with Tt <= Tp: loss over pred[:, :Tt]
  const int64_t n = B * Tt * C;
  const float inv_n = 1.f / (float)n;
  float local = 0.f;
  const int64_t total = B * Tp * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = i % C, t = (i / C) % Tp, b = i / (C * Tp);
    float g = 0.f;
    if (t < Tt) {
      const int64_t j = (b * Tt + t) * C + c;
      const float tv = tgt_f ? tgt_f[j] : (float)tgt_i[j];
      const float d = pred[i] - tv;
      local += fabsf(d);
      g = (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f)) * weight * inv_n;
    }
    if (grad) grad[i] = g;
  }
  local = wsum(local);
  __shared__ float red[32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    atomicAdd(loss_out, s * inv_n);
  }
}

// ------------------------------------------------------------------------------------------------
// Aligner losses (SURVEY 8(f) row 1)
//   scaled_ce: utils/losses.py:4-21 -- sparse softmax cross entropy of logits (B,Tp,C)[:, :Tt] vs int targets (B,Tt),
//     weight = (target != 0) + (target == index) * (scaling - 1), Keras SUM_OVER_BATCH_SIZE: sum / (B*Tt)
//   diag_loss: utils/metrics.py:47-70 + models.py:189-205 -- mean over (b,h) of sum_{q,k} att * |k/k_len - q/q_len| / 10
// ------------------------------------------------------------------------------------------------
__global__ void scaled_ce_kernel(const float* __restrict__ logits, int64_t B, int64_t Tp, int64_t Tt, int C, int ld,
                                 const int* __restrict__ tgt, int index, float scaling, float* __restrict__ loss_out,
                                 float grad_weight, float* __restrict__ grad, int ld_grad) {
  const int64_t n = B * Tt;
  float local = 0.f;
  // rows of the prediction beyond the target length (t >= Tt) carry no loss: zero gradient
  const int64_t total = grad ? B * Tp : n;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = grad ? i / Tp : i / Tt, t = grad ? i % Tp : i % Tt;
    if (t >= Tt) {
      for (int c = 0; c < C; ++c) grad[(b * Tp + t) * ld_grad + c] = 0.f;
      continue;
    }
    const float* row = logits + (b * Tp + t) * ld;
    const int y = tgt[b * Tt + t];
    float mx = row[0];
    for (int c = 1; c < C; ++c) mx = fmaxf(mx, row[c]);
    float se = 0.f;
    for (int c = 0; c < C; ++c) se += expf(row[c] - mx);
    const float ce = (y >= 0 && y < C) ? (logf(se) + mx - row[y]) : 0.f;
    const float w = (y != 0 ? 1.f : 0.f) + (y == index ? scaling - 1.f : 0.f);
    local += ce * w;
    if (grad) {
      const float gs = grad_weight * w / (float)n;
      for (int c = 0; c < C; ++c) grad[(b * Tp + t) * ld_grad + c] = gs * (expf(row[c] - mx) / se - (c == y ? 1.f : 0.f));
    }
  }
  local = wsum(local);
  __shared__ float red[32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    atomicAdd(loss_out, s / (float)n);
  }
}

__global__ void diag_loss_kernel(const float* __restrict__ att, int H, int Tq, int Tk, const int* __restrict__ q_len,
                                 const int* __restrict__ k_len, float scale, float* __restrict__ loss_out) {
  // grid (B*H, ceil(Tq / 32)): one warp per query row, lanes across the keys
  const int bh = blockIdx.x;
  const int b = bh / H;
  const int max_m = min(max(q_len[b], 0), Tq);  // metrics.py:62-64
  const int max_n = min(max(k_len[b], 0), Tk);
  const float* a = att + (size_t)bh * Tq * Tk;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float local = 0.f;
  const int q_end = min(max_m, (int)(blockIdx.y + 1) * 32);
  for (int q = blockIdx.y * 32 + wid; q < q_end; q += nw) {
    const double jq = (double)q / (double)max_m;
    for (int k = lane; k < max_n; k += 32) {
      // the reference divides int32 ranges (-> float64), takes |.|, then casts the mask to float32
      const float m = (float)fabs((double)k / (double)max_n - jq);
      local += a[(size_t)q * Tk + k] * m;
    }
  }
  local = wsum(local);
  __shared__ float red[32];
  if (lane == 0) red[wid] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < nw; ++w) s += red[w];
    if (s != 0.f) atomicAdd(loss_out, s * scale);
  }
}

// training form of the diagonal loss: the maps are the post-dropout probabilities P (bf16, (B*H, Tq, ld)); the loss is
// added to *loss_out (scaled by loss_scale / (10*B*H)) and its gradient grad_scale / (10*B*H) * mask is added to dP (fp32,
// same layout), the gradient of the P.V product, before the softmax backward.
__global__ void diag_loss_train_kernel(const __nv_bfloat16* __restrict__ P, int H, int Tq, int Tk, int ld, const int* __restrict__ q_len,
                                       const int* __restrict__ k_len, float loss_scale, float* __restrict__ loss_out, float grad_scale,
                                       float* __restrict__ dP) {
  const int bh = blockIdx.x;
  const int b = bh / H;
  const int max_m = min(max(q_len[b], 0), Tq);
  const int max_n = min(max(k_len[b], 0), Tk);
  const size_t base = (size_t)bh * Tq * ld;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float local = 0.f;
  const int q_end = min(max_m, (int)(blockIdx.y + 1) * 32);
  for (int q = blockIdx.y * 32 + wid; q < q_end; q += nw) {
    const double jq = (double)q / (double)max_m;
    for (int k = lane; k < max_n; k += 32) {
      const float m = (float)fabs((double)k / (double)max_n - jq);
      const size_t i = base + (size_t)q * ld + k;
      local += __bfloat162float(P[i]) * m;
      if (dP) dP[i] += grad_scale * m;
    }
  }
  local = wsum(local);
  __shared__ float red[32];
  if (lane == 0) red[wid] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < nw; ++w) s += red[w];
    if (s != 0.f) atomicAdd(loss_out, s * loss_scale);
  }
}

// ------------------------------------------------------------------------------------------------
// D[(b*H + h)*T + t] = sum_c x[b,t,h*dh+c] * y[b,t,h*dh+c]   (one warp per (b,t) row, heads in sequence)
// ------------------------------------------------------------------------------------------------
__global__ void rowdot_heads_kernel(const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ y, int rows, int T, int H,
                                    int dh, int ld, float* __restrict__ out) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int b = row / T, t = row % T;
  const __nv_bfloat162* xr = reinterpret_cast<const __nv_bfloat162*>(x + (size_t)row * ld);
  const __nv_bfloat162* yr = reinterpret_cast<const __nv_bfloat162*>(y + (size_t)row * ld);
  for (int h = 0; h < H; ++h) {
    float acc = 0.f;
    for (int c = lane; c < dh / 2; c += 32) {
      const float2 a = __bfloat1622float2(xr[h * (dh / 2) + c]);
      const float2 v = __bfloat1622float2(yr[h * (dh / 2) + c]);
      acc = fmaf(a.x, v.x, fmaf(a.y, v.y, acc));
    }
    acc = wsum(acc);
    if (lane == 0) out[((size_t)b * H + h) * T + t] = acc;
  }
}

// ------------------------------------------------------------------------------------------------
// Expand backward: dx[b,i,:] = sum of dm[b, t, :] over the frames t copied from phoneme i (contiguous segment)
// ------------------------------------------------------------------------------------------------
__global__ void expand_bwd_kernel(const float* __restrict__ dm, const int* __restrict__ dur, int Tp, int Tm, int d,
                                  float* __restrict__ dx) {
  // grid (B, chunks): every block rebuilds the row's exclusive prefix sum with a block scan, then its warps take the phoneme
  // segments of its chunk; a lane owns float4 columns, the frame loop is unrolled by two for memory-level parallelism.
  extern __shared__ int cum[];  // exclusive starts, Tp+1
  __shared__ int wtot[32];
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  int carry = 0;
  for (int base = 0; base < Tp; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const int v = i < Tp ? max(dur[(size_t)b * Tp + i], 0) : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += u;
    }
    if (lane == 31) wtot[warp] = incl;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < warp; ++w) woff += wtot[w];
    if (i < Tp) cum[i] = carry + woff + incl - v;
    int tot = 0;
    for (int w = 0; w < warps; ++w) tot += wtot[w];
    carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) cum[Tp] = carry;
  __syncthreads();
  const int d4 = d >> 2;
  for (int i = blockIdx.y * warps + warp; i < Tp; i += gridDim.y * warps) {
    const int s = min(cum[i], Tm), e = min(cum[i + 1], Tm);
    const float4* src = reinterpret_cast<const float4*>(dm + ((size_t)b * Tm) * d);
    for (int c = lane; c < d4; c += 32) {
      float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
      int t = s;
      for (; t + 1 < e; t += 2) {
        const float4 u = src[(size_t)t * d4 + c], v = src[(size_t)(t + 1) * d4 + c];
        a0.x += u.x; a0.y += u.y; a0.z += u.z; a0.w += u.w;
        a1.x += v.x; a1.y += v.y; a1.z += v.z; a1.w += v.w;
      }
      if (t < e) {
        const float4 u = src[(size_t)t * d4 + c];
        a0.x += u.x; a0.y += u.y; a0.z += u.z; a0.w += u.w;
      }
      reinterpret_cast<float4*>(dx + ((size_t)b * Tp + i) * d)[c] = make_float4(a0.x + a1.x, a0.y + a1.y, a0.z + a1.z, a0.w + a1.w);
    }
  }
}

__global__ void embedding_bwd_kernel(const float* __restrict__ dx, const int* __restrict__ tokens, int rows, int d, int vocab,
                                     float* __restrict__ demb) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  int tok = tokens[row];
  tok = tok < 0 ? 0 : (tok >= vocab ? vocab - 1 : tok);
  for (int c = threadIdx.x & 31; c < d; c += 32) atomicAdd(demb + (size_t)tok * d + c, dx[(size_t)row * d + c]);
}

// positional-encoding scalar gradient: sum_{row,c} g[row,c] * pe[t,c]   (d % 4 == 0: float4 columns, 32-bit index math)
__global__ void pe_scalar_bwd_kernel(const float* __restrict__ g, const float* __restrict__ pe, int rows, int T, int d,
                                     float drop_p, uint32_t seed, uint32_t site, float* __restrict__ dscalar) {
  const uint32_t thresh = dropout_thresh(drop_p);
  const float keep_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  float local = 0.f;
  const int d4 = d >> 2;
  const int rpb = blockDim.x / d4 > 0 ? blockDim.x / d4 : 1;        // rows a block covers per sweep (d4 <= blockDim.x)
  const int c4 = threadIdx.x % d4, rsub = threadIdx.x / d4;
  if (rsub < rpb) {
    for (int row = blockIdx.x * rpb + rsub; row < rows; row += gridDim.x * rpb) {
      const int t = row % T;
      float4 gv = reinterpret_cast<const float4*>(g + (size_t)row * d)[c4];
      const float4 pv = __ldg(reinterpret_cast<const float4*>(pe + (size_t)t * d) + c4);
      if (drop_p > 0.f) {
        const uint64_t i0 = (uint64_t)row * d + 4 * c4;
        bool k0, k1, k2, k3;
        dropout_keep2(seed, site, i0, thresh, k0, k1);
        dropout_keep2(seed, site, i0 + 2, thresh, k2, k3);
        gv.x = k0 ? gv.x * keep_scale : 0.f; gv.y = k1 ? gv.y * keep_scale : 0.f;
        gv.z = k2 ? gv.z * keep_scale : 0.f; gv.w = k3 ? gv.w * keep_scale : 0.f;
      }
      local = fmaf(gv.x, pv.x, fmaf(gv.y, pv.y, fmaf(gv.z, pv.z, fmaf(gv.w, pv.w, local))));
    }
  }
  local = wsum(local);
  __shared__ float red[32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    atomicAdd(dscalar, s);
  }
}

// the same for widths that are not a multiple of four (or wider than a block)
__global__ void pe_scalar_bwd_scalar_kernel(const float* __restrict__ g, const float* __restrict__ pe, int rows, int T, int d,
                                            float drop_p, uint32_t seed, uint32_t site, float* __restrict__ dscalar) {
  const uint32_t thresh = dropout_thresh(drop_p);
  const float keep_scale = drop_p > 0.f ? 1.f / (1.f - drop_p) : 1.f;
  float local = 0.f;
  const int64_t n = (int64_t)rows * d;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % d);
    const int t = (int)((i / d) % T);
    float gv = g[i];
    if (drop_p > 0.f) gv = dropout_keep(seed, site, (uint64_t)i, thresh) ? gv * keep_scale : 0.f;
    local += gv * __ldg(pe + (size_t)t * d + c);
  }
  local = wsum(local);
  __shared__ float red[32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    atomicAdd(dscalar, s);
  }
}

// pitch embedding Dense(1->d, relu) gradients w.r.t. its kernel and bias: pre = pitch*w + b.  Threads run along the
// channels (coalesced rows of g); a block takes a 64-row slab and folds its partial sums with one atomic per channel.
__global__ void pitch_embed_bwd_kernel(const float* __restrict__ g, const float* __restrict__ pitch, const float* __restrict__ w,
                                       const float* __restrict__ bias, int rows, int d, float* __restrict__ dw, float* __restrict__ db) {
  const int r0 = blockIdx.x * 64, r1 = min(r0 + 64, rows);
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    const float wc = w[c], bc = bias[c];
    float sw = 0.f, sb = 0.f;
#pragma unroll 4
    for (int r = r0; r < r1; ++r) {
      const float pv = __ldg(pitch + r);
      const float gv = g[(size_t)r * d + c];
      if (fmaf(pv, wc, bc) > 0.f) { sw = fmaf(gv, pv, sw); sb += gv; }
    }
    atomicAdd(dw + c, sw);
    atomicAdd(db + c, sb);
  }
}

// StatPredictor head backward: out = act(h.w + b) * mask
__global__ void statpred_head_bwd_kernel(const float* __restrict__ gout, const float* __restrict__ out, const float* __restrict__ h,
                                         int ldh, int C, const float* __restrict__ w, int relu, const int* __restrict__ row_len,
                                         int rows, int T, float* __restrict__ dh, float* __restrict__ dw, float* __restrict__ db) {
  extern __shared__ float part[];  // C + 1
  for (int c = threadIdx.x; c <= C; c += blockDim.x) part[c] = 0.f;
  __syncthreads();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row < rows) {
    const int b = row / T, t = row % T;
    float g = gout[row];
    if (row_len && t >= row_len[b]) g = 0.f;
    if (relu && !(out[row] > 0.f)) g = 0.f;
    for (int c = lane; c < ldh; c += 32) {
      float v = 0.f;
      if (c < C) {
        v = g * __ldg(w + c);
        if (g != 0.f) atomicAdd(part + c, g * h[(size_t)row * ldh + c]);
      }
      dh[(size_t)row * ldh + c] = v;
    }
    if (lane == 0 && g != 0.f) atomicAdd(part + C, g);
  }
  __syncthreads();
  for (int c = threadIdx.x; c <= C; c += blockDim.x)
    if (part[c] != 0.f) atomicAdd(c < C ? dw + c : db, part[c]);
}

// Keras (TF 2.2) Adam: theta -= lr_t * m / (sqrt(v) + eps), lr_t = lr*sqrt(1-b2^t)/(1-b1^t) computed by the host
__global__ void adam_tf_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                               int64_t n, float lr_t, float b1, float b2, float eps, float gscale) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i] * gscale;
  const float mi = b1 * m[i] + (1.f - b1) * gi;
  const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  p[i] -= lr_t * mi / (sqrtf(vi) + eps);
}

static inline int bad(const char* msg) {
  set_last_error("%s", msg);
  return TTSB_ERR_INVALID_ARGUMENT;
}

}  // namespace ttsb

using namespace ttsb;
#define STREAM(s) static_cast<cudaStream_t>(s)
#define LAUNCH_OK(name) \
  count_launch();       \
  return check_cuda(cudaGetLastError(), name)
#define BF(p) static_cast<__nv_bfloat16*>(p)
#define CBF(p) static_cast<const __nv_bfloat16*>(p)

extern "C" int ttsb_softmax_fwd(const float* S, int B, int H, int T, int Tk, int ld, const int32_t* kv_len, float drop_p,
                                uint32_t seed, uint32_t site, int flags, void* P_pre, void* P_drop, void* stream) {
  if (!S || !kv_len || !P_pre || !P_drop || B <= 0 || H <= 0 || T <= 0 || Tk <= 0 || ld < Tk) return bad("ttsb_softmax_fwd: bad arguments");
  const int rows = B * H * T;
  if (ld % 4 == 0 && ld <= 1024 && (reinterpret_cast<uintptr_t>(S) & 15) == 0 && (reinterpret_cast<uintptr_t>(P_pre) & 7) == 0 &&
      (reinterpret_cast<uintptr_t>(P_drop) & 7) == 0) {
#define TTSB_SMV(NG)                                                                                                                  \
  softmax_fwd_vec_kernel<NG><<<(rows + 7) / 8, 256, 0, STREAM(stream)>>>(S, B * H, H, T, Tk, ld, kv_len, drop_p, seed, site, flags, \
                                                                          BF(P_pre), BF(P_drop))
    if (ld <= 128) TTSB_SMV(1);
    else if (ld <= 256) TTSB_SMV(2);
    else if (ld <= 512) TTSB_SMV(4);
    else TTSB_SMV(8);
#undef TTSB_SMV
    LAUNCH_OK("softmax_fwd_vec_kernel");
  }
  softmax_fwd_kernel<<<(rows + 7) / 8, 256, 0, STREAM(stream)>>>(S, B * H, H, T, Tk, ld, kv_len, drop_p, seed, site, flags, BF(P_pre), BF(P_drop));
  LAUNCH_OK("softmax_fwd_kernel");
}

extern "C" int ttsb_softmax_bwd(const void* P_pre, const float* dP, int B, int H, int T, int Tk, int ld, const int32_t* kv_len,
                                float scale, float drop_p, uint32_t seed, uint32_t site, int flags, void* dS, void* stream) {
  if (!P_pre || !dP || !kv_len || !dS || B <= 0 || H <= 0 || T <= 0 || Tk <= 0 || ld < Tk) return bad("ttsb_softmax_bwd: bad arguments");
  const int rows = B * H * T;
  softmax_bwd_kernel<<<(rows + 7) / 8, 256, 0, STREAM(stream)>>>(CBF(P_pre), dP, B * H, H, T, Tk, ld, kv_len, scale, drop_p, seed, site, flags, BF(dS));
  LAUNCH_OK("softmax_bwd_kernel");
}

extern "C" int ttsb_layernorm_bwd(const float* dz, const float* u, const float* gamma, int B, int T, int C, int ld, float eps,
                                  const int32_t* row_len, int relu_mask, float pre_drop_p, uint32_t pre_site, float post_drop_p,
                                  uint32_t post_site, uint32_t seed, float* du, void* g_bf16, float* dgamma, float* dbeta, float* dbias,
                                  void* stream) {
  if (!dz || !u || !gamma || !dgamma || !dbeta || B <= 0 || T <= 0 || C <= 0 || C > 512 || ld < C || ld > 512)
    return bad("ttsb_layernorm_bwd: bad arguments (C, ld <= 512)");
  const int rows = B * T;
  if (C == ld && C % 128 == 0 && C <= 384 && (long long)rows * C < (1ll << 33)) {   // every block LayerNorm of the model: vectorised persistent kernel
    const int grid = min((rows + 7) / 8, 2 * num_sms());
#define TTSB_LNV(NG)                                                                                                            \
  layernorm_bwd_vec_kernel<NG><<<grid, 256, 0, STREAM(stream)>>>(dz, u, gamma, rows, T, eps, row_len, relu_mask, pre_drop_p, pre_site, \
                                                                post_drop_p, post_site, seed, du, BF(g_bf16), dgamma, dbeta, dbias)
    if (C == 128) TTSB_LNV(1);
    else if (C == 256) TTSB_LNV(2);
    else TTSB_LNV(3);
#undef TTSB_LNV
    LAUNCH_OK("layernorm_bwd_vec_kernel");
  }
  const int blocks = (rows + 31) / 32;
  const size_t sm = 3 * C * sizeof(float);
#define TTSB_LNB(NV)                                                                                                              \
  layernorm_bwd_kernel<NV><<<blocks, 256, sm, STREAM(stream)>>>(dz, u, gamma, rows, T, C, ld, eps, row_len, relu_mask, pre_drop_p, \
                                                                 pre_site, post_drop_p, post_site, seed, du, BF(g_bf16), dgamma, dbeta, dbias)
  if (ld <= 128) TTSB_LNB(4);
  else if (ld <= 256) TTSB_LNB(8);
  else if (ld <= 384) TTSB_LNB(12);
  else TTSB_LNB(16);
#undef TTSB_LNB
  LAUNCH_OK("layernorm_bwd_kernel");
}

extern "C" int ttsb_colsum_bf16(const void* x, int64_t rows, int C, int ld, float* out, void* stream) {
  if (!x || !out || rows <= 0 || C <= 0 || ld < C || ld % 8 || (ld < ((C + 7) / 8) * 8)) return bad("ttsb_colsum_bf16: need ld % 8 == 0 and ld >= round_up(C, 8)");
  dim3 grid((C + 255) / 256, (unsigned)((rows + 127) / 128));
  colsum_bf16_kernel<<<grid, 256, 0, STREAM(stream)>>>(CBF(x), rows, C, ld, out, C, nullptr, nullptr);
  LAUNCH_OK("colsum_bf16_kernel");
}

extern "C" int ttsb_colsum_bf16_x3(const void* x, int64_t rows, int seg, int ld, float* out0, float* out1, float* out2, void* stream) {
  if (!x || !out0 || !out1 || !out2 || rows <= 0 || seg <= 0 || seg % 8 || ld < 3 * seg || ld % 8)
    return bad("ttsb_colsum_bf16_x3: need seg % 8 == 0 and ld >= 3 * seg, ld % 8 == 0");
  dim3 grid((3 * seg + 255) / 256, (unsigned)((rows + 127) / 128));
  colsum_bf16_kernel<<<grid, 256, 0, STREAM(stream)>>>(CBF(x), rows, 3 * seg, ld, out0, seg, out1, out2);
  LAUNCH_OK("colsum_bf16_kernel");
}

extern "C" int ttsb_relu_bwd(void* dy, const void* h, int64_t n, void* stream) {
  if (!dy || !h || n <= 0 || n % 8) return bad("ttsb_relu_bwd: n must be a positive multiple of 8");
  relu_bwd_kernel<<<(unsigned)((n / 8 + 255) / 256), 256, 0, STREAM(stream)>>>(BF(dy), CBF(h), n);
  LAUNCH_OK("relu_bwd_kernel");
}

extern "C" int ttsb_relu_bwd_colsum(void* dy, const void* h, int64_t rows, int C, float* colsum, void* stream) {
  if (!dy || !h || !colsum || rows <= 0 || C <= 0 || C % 8) return bad("ttsb_relu_bwd_colsum: C must be a positive multiple of 8");
  dim3 grid((C + 255) / 256, (unsigned)((rows + 127) / 128));
  relu_bwd_colsum_kernel<<<grid, 256, 0, STREAM(stream)>>>(BF(dy), CBF(h), rows, C, colsum);
  LAUNCH_OK("relu_bwd_colsum_kernel");
}

extern "C" int ttsb_cast_bf16_pad(const float* x, int64_t rows, int C, void* out, int ld_out, void* stream) {
  if (!x || !out || rows <= 0 || C <= 0 || ld_out < C) return bad("ttsb_cast_bf16_pad: bad arguments");
  const int64_t n = rows * ld_out;
  cast_bf16_pad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, STREAM(stream)>>>(x, rows, C, BF(out), ld_out);
  LAUNCH_OK("cast_bf16_pad_kernel");
}

extern "C" int ttsb_mae_loss(const float* pred, int B, int Tp, int Tt, int C, const float* target_f32, const int32_t* target_i32,
                             float weight, float* loss_out, float* grad, void* stream) {
  if (!pred || (!target_f32 && !target_i32) || !loss_out || B <= 0 || Tp <= 0 || Tt <= 0 || Tt > Tp || C <= 0)
    return bad("ttsb_mae_loss: bad arguments (need Tt <= Tp)");
  mae_loss_kernel<<<592, 256, 0, STREAM(stream)>>>(pred, B, Tp, Tt, C, target_f32, target_i32, weight, loss_out, grad);
  LAUNCH_OK("mae_loss_kernel");
}

extern "C" int ttsb_scaled_ce_loss(const float* logits, int B, int Tp, int Tt, int C, int ld, const int32_t* targets, int index,
                                   float scaling, float* loss_out, float grad_weight, float* grad, int ld_grad, void* stream) {
  if (!logits || !targets || !loss_out || B <= 0 || Tp <= 0 || Tt <= 0 || Tt > Tp || C <= 0 || ld < C || (grad && ld_grad < C))
    return bad("ttsb_scaled_ce_loss: bad arguments (need Tt <= Tp, ld >= C)");
  scaled_ce_kernel<<<148, 256, 0, STREAM(stream)>>>(logits, B, Tp, Tt, C, ld, targets, index, scaling, loss_out, grad_weight, grad, ld_grad);
  LAUNCH_OK("scaled_ce_kernel");
}

extern "C" int ttsb_diag_loss(const float* att, int B, int H, int Tq, int Tk, const int32_t* q_len, const int32_t* k_len,
                              float* loss_out, void* stream) {
  if (!att || !q_len || !k_len || !loss_out || B <= 0 || H <= 0 || Tq <= 0 || Tk <= 0) return bad("ttsb_diag_loss: bad arguments");
  diag_loss_kernel<<<dim3(B * H, (Tq + 31) / 32), 256, 0, STREAM(stream)>>>(att, H, Tq, Tk, q_len, k_len, 1.f / (10.f * (float)(B * H)), loss_out);
  LAUNCH_OK("diag_loss_kernel");
}

extern "C" int ttsb_diag_loss_train(const void* P_bf16, int B, int H, int Tq, int Tk, int ld, const int32_t* q_len,
                                    const int32_t* k_len, float loss_scale, float* loss_out, float grad_scale, float* dP, void* stream) {
  if (!P_bf16 || !q_len || !k_len || !loss_out || B <= 0 || H <= 0 || Tq <= 0 || Tk <= 0 || ld < Tk) return bad("ttsb_diag_loss_train: bad arguments");
  const float inv = 1.f / (10.f * (float)(B * H));
  diag_loss_train_kernel<<<dim3(B * H, (Tq + 31) / 32), 256, 0, STREAM(stream)>>>(CBF(P_bf16), H, Tq, Tk, ld, q_len, k_len, loss_scale * inv,
                                                                                  loss_out, grad_scale * inv, dP);
  LAUNCH_OK("diag_loss_train_kernel");
}

extern "C" int ttsb_rowdot_heads(const void* x, const void* y, int B, int T, int H, int dh, int ld, float* out, void* stream) {
  if (!x || !y || !out || B <= 0 || T <= 0 || H <= 0 || dh <= 0 || dh % 2 || ld < H * dh || ld % 2) return bad("ttsb_rowdot_heads: bad arguments");
  const int rows = B * T;
  rowdot_heads_kernel<<<(rows + 7) / 8, 256, 0, STREAM(stream)>>>(CBF(x), CBF(y), rows, T, H, dh, ld, out);
  LAUNCH_OK("rowdot_heads_kernel");
}

extern "C" int ttsb_expand_bwd(const float* dm, const int32_t* dur_int, int B, int Tp, int Tm, int d, float* dx, void* stream) {
  if (!dm || !dur_int || !dx || B <= 0 || Tp <= 0 || Tm <= 0 || d <= 0) return bad("ttsb_expand_bwd: bad arguments");
  // the kernel walks rows as float4 columns: dm / dx rows start 16-byte aligned only when d % 4 == 0
  if (d % 4 || (reinterpret_cast<uintptr_t>(dm) & 15) || (reinterpret_cast<uintptr_t>(dx) & 15))
    return bad("ttsb_expand_bwd: d must be a multiple of 4 and dm, dx 16-byte aligned");
  const int chunks = std::min(32, (Tp + 7) / 8);
  expand_bwd_kernel<<<dim3(B, chunks), 256, (Tp + 1) * sizeof(int), STREAM(stream)>>>(dm, dur_int, Tp, Tm, d, dx);
  LAUNCH_OK("expand_bwd_kernel");
}

extern "C" int ttsb_embedding_bwd(const float* dx, const int32_t* tokens, int B, int T, int d, int vocab, float* demb, void* stream) {
  if (!dx || !tokens || !demb || B <= 0 || T <= 0 || d <= 0 || vocab <= 0) return bad("ttsb_embedding_bwd: bad arguments");
  const int rows = B * T;
  embedding_bwd_kernel<<<(rows + 7) / 8, 256, 0, STREAM(stream)>>>(dx, tokens, rows, d, vocab, demb);
  LAUNCH_OK("embedding_bwd_kernel");
}

extern "C" int ttsb_pe_scalar_bwd(const float* g, const float* pe, int B, int T, int d, float drop_p, uint32_t seed, uint32_t site,
                                  float* dscalar, void* stream) {
  if (!g || !pe || !dscalar || B <= 0 || T <= 0 || d <= 0) return bad("ttsb_pe_scalar_bwd: bad arguments");
  if (d % 4 == 0 && d / 4 <= 384)
    pe_scalar_bwd_kernel<<<592, 384, 0, STREAM(stream)>>>(g, pe, B * T, T, d, drop_p, seed, site, dscalar);
  else
    pe_scalar_bwd_scalar_kernel<<<296, 256, 0, STREAM(stream)>>>(g, pe, B * T, T, d, drop_p, seed, site, dscalar);
  LAUNCH_OK("pe_scalar_bwd_kernel");
}

extern "C" int ttsb_pitch_embed_bwd(const float* g, const float* pitch, const float* w, const float* bias, int B, int T, int d,
                                    float* dw, float* db, void* stream) {
  if (!g || !pitch || !w || !bias || !dw || !db || B <= 0 || T <= 0 || d <= 0) return bad("ttsb_pitch_embed_bwd: bad arguments");
  const int rows = B * T;
  pitch_embed_bwd_kernel<<<(rows + 63) / 64, std::min(512, ((d + 31) / 32) * 32), 0, STREAM(stream)>>>(g, pitch, w, bias, rows, d, dw, db);
  LAUNCH_OK("pitch_embed_bwd_kernel");
}

extern "C" int ttsb_statpred_head_bwd(const float* gout, const float* out, const float* h, int ldh, int C, const float* w, int relu,
                                      const int32_t* row_len, int B, int T, float* dh, float* dw, float* db, void* stream) {
  if (!gout || !out || !h || !w || !dh || !dw || !db || B <= 0 || T <= 0 || C <= 0 || ldh < C) return bad("ttsb_statpred_head_bwd: bad arguments");
  const int rows = B * T;
  statpred_head_bwd_kernel<<<(rows + 7) / 8, 256, (C + 1) * sizeof(float), STREAM(stream)>>>(gout, out, h, ldh, C, w, relu, row_len, rows, T, dh, dw, db);
  LAUNCH_OK("statpred_head_bwd_kernel");
}

extern "C" int ttsb_adam_tf_step(float* param, const float* grad, float* m, float* v, int64_t n, float lr_t, float beta1, float beta2,
                                 float eps, float grad_scale, void* stream) {
  if (!param || !grad || !m || !v || n <= 0) return bad("ttsb_adam_tf_step: bad arguments");
  adam_tf_kernel<<<(unsigned)((n + 255) / 256), 256, 0, STREAM(stream)>>>(param, grad, m, v, n, lr_t, beta1, beta2, eps, grad_scale);
  LAUNCH_OK("adam_tf_kernel");
}

TTSB_DEFINE_SALT_SETTER(set_salt_train_ops)
