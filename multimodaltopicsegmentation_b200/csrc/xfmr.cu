// Pyramidal windowed-attention encoder, forward kernels.  Restates what the reference obtains from HF
// `LongformerModel(inputs_embeds=...)` (models/RestrictedTransformerLayer.py:65-133 -> HF modeling_longformer.py):
//   * LongformerEmbeddings (:401-442): LN_{eps}(x + P[2 + t] + E_type[0])            -> mts_embed_ln_fwd
//   * LongformerSelfOutput / LongformerOutput (:1060-1071, :1119-1130): LN(dense + x) -> mts_add_ln_fwd
//   * LongformerSelfAttention (:481-639, sliding chunks :758-867): softmax over |i-j| <= w, j < len_b,
//     q scaled by 1/sqrt(hd), masked queries output exact zeros                    -> mts_band_attn_fwd
//   * LongformerIntermediate (:1103-1116): GELU(erf); fused here with the hi/lo split that feeds the
//     next 3xTF32 GEMM                                                              -> mts_gelu_split
// No mask tensor is ever built (create_masks_huggingface, RestrictedTransformerLayer.py:101-116, is a host
// double loop in the reference): every kernel takes `lengths`.
//
// The dense layers themselves are mts_gemm_tf32x3 (tcgen05).  The kernels here are the HBM-bound glue:
// LN kernels move 4d in + 4d (+ 8 Kp for the GEMM operand halves) out per token; the attention kernel reads
// q,k,v (12d) and writes o (4d, or the two operand halves) per token and only ever touches in-window keys.
#include <stdlib.h>

#include <cuda_fp16.h>

#include "common.cuh"

namespace mts {

// ---------------------------------------------------------------------------------------------------------
// LayerNorm forward, one warp per token row, values held in registers (two-pass mean / variance).
//   MODE 0: v = x[b, t, :] + pos[t + 2, :] + typ[:]       (embeddings; position ids start at pad_token_id + 1 = 2)
//   MODE 1: v = a[row, :] + res[row, :]                    (dense output + residual)
//   MODE 2: MODE 0 with x given as bf16                    (embeddings stored and shipped in bf16: half the host-to-device bytes)
// outputs: y fp32, optional (hi, lo) TF32 halves [M, Kp] for the next GEMM, optional pre-LN sum and
// (mean, rstd) for the backward pass.
// ---------------------------------------------------------------------------------------------------------
constexpr int LN_MAXV = 16;  // float4 per lane -> d <= 2048 (MAXV = 8 serves d <= 1024 with half the registers)

// PIECES: instead of the (hi, lo) pair the kernel writes the fp16-split operand of mts_gemm_f16x3 -- y_lo then points to
// __half pieces [M][2][Kp] (Kp a multiple of 64: fp16 elements) and row_scale [M] receives 2^-s, where 2^s is the exact
// power of two that puts the row's largest |y| into [2^13, 2^14) (a warp owns a row, so its maximum is one shuffle tree away).
template <int MODE, int MAXV, bool PIECES = false>
__global__ void __launch_bounds__(256) ln_fwd_kernel(const float *__restrict__ a, int64_t a_bstride,
                                                     const float *__restrict__ b, const float *__restrict__ typ,
                                                     const float *__restrict__ gamma, const float *__restrict__ beta,
                                                     int M, int S, int d, float eps, float *__restrict__ y,
                                                     float *__restrict__ y_hi, float *__restrict__ y_lo, int Kp,
                                                     float *__restrict__ sum_out, float *__restrict__ stats,
                                                     const int32_t *__restrict__ lengths,
                                                     const int32_t *__restrict__ offsets, float *__restrict__ row_scale = nullptr) {
  const int lane = threadIdx.x & 31;
  const int nv = d >> 2;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int in_row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; in_row < M; in_row += warps) {
    const float4 *pa, *pb;
    int row = in_row;
    if (MODE != 1) {
      const int bi = in_row / S, t = in_row % S;
      if (offsets) {  // ragged output: valid sentences only, episode bi starts at row offsets[bi]
        if (t >= lengths[bi]) continue;
        row = offsets[bi] + t;
      }
      if (MODE == 2)   // 4 bf16 (8 bytes) per float4 column: pa is only a row address here, read as uint2 below
        pa = reinterpret_cast<const float4 *>(reinterpret_cast<const uint16_t *>(a) + (int64_t)bi * a_bstride + (int64_t)t * d);
      else
        pa = reinterpret_cast<const float4 *>(a + (int64_t)bi * a_bstride + (int64_t)t * d);
      pb = reinterpret_cast<const float4 *>(b + (int64_t)(t + 2) * d);
    } else {
      pa = reinterpret_cast<const float4 *>(a + (int64_t)row * d);
      pb = b ? reinterpret_cast<const float4 *>(b + (int64_t)row * d) : nullptr;  // null: `a` already holds the sum
    }
    // float4 column of register i: lanes own PAIRS of adjacent float4 (8 consecutive elements), so that the packed
    // correction operand goes out in 16-byte pieces (corr_store8)
#define LN_COL(i) (2 * (lane + 32 * ((i) >> 1)) + ((i) & 1))
    float4 v[MAXV];
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int c = LN_COL(i);
      if (c < nv) {
        float4 x;
        if (MODE == 2) {
          const uint2 u = __ldg(reinterpret_cast<const uint2 *>(pa) + c);
          x = make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xFFFF0000u), __uint_as_float(u.y << 16),
                          __uint_as_float(u.y & 0xFFFF0000u));
        } else {
          x = __ldg(pa + c);
        }
        if (MODE != 1 || pb) {
          const float4 r = __ldg(pb + c);
          x.x += r.x; x.y += r.y; x.z += r.z; x.w += r.w;
        }
        if (MODE != 1) {
          const float4 e = __ldg(reinterpret_cast<const float4 *>(typ) + c);
          x.x += e.x; x.y += e.y; x.z += e.z; x.w += e.w;
        }
        v[i] = x;
        s += (x.x + x.y) + (x.z + x.w);
      }
    }
    const float mean = warp_sum(s) / (float)d;
    float q = 0.0f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      if (LN_COL(i) < nv) {
        const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
        q += (dx * dx + dy * dy) + (dz * dz + dw * dw);
      }
    }
    const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)d + eps);
    if (stats && lane == 0) { stats[2 * (int64_t)row] = mean; stats[2 * (int64_t)row + 1] = rstd; }
    if (PIECES) {
      // normalised values in place, the row's largest magnitude, its power-of-two scale, then y and the two fp16 pieces
      float mx = 0.0f;
#pragma unroll
      for (int i = 0; i < MAXV; ++i) {
        const int c = LN_COL(i);
        if (c < nv) {
          if (sum_out) reinterpret_cast<float4 *>(sum_out + (int64_t)row * d)[c] = v[i];
          const float4 g = __ldg(reinterpret_cast<const float4 *>(gamma) + c);
          const float4 be = __ldg(reinterpret_cast<const float4 *>(beta) + c);
          v[i].x = (v[i].x - mean) * rstd * g.x + be.x;
          v[i].y = (v[i].y - mean) * rstd * g.y + be.y;
          v[i].z = (v[i].z - mean) * rstd * g.z + be.z;
          v[i].w = (v[i].w - mean) * rstd * g.w + be.w;
          reinterpret_cast<float4 *>(y + (int64_t)row * d)[c] = v[i];
          mx = fmaxf(fmaxf(mx, fmaxf(fabsf(v[i].x), fabsf(v[i].y))), fmaxf(fabsf(v[i].z), fabsf(v[i].w)));
        }
      }
      mx = warp_max(mx);
      const int ex = (int)((__float_as_uint(mx) >> 23) & 0xFFu);
      int sexp = ex == 0 ? 0 : 127 + 13 - ex;
      sexp = sexp > 110 ? 110 : (sexp < -110 ? -110 : sexp);
      const float sc = __uint_as_float((uint32_t)(127 + sexp) << 23);
      if (lane == 0) row_scale[row] = __uint_as_float((uint32_t)(127 - sexp) << 23);
      __half *p1 = reinterpret_cast<__half *>(y_lo) + (int64_t)row * 2 * Kp, *p2 = p1 + Kp;
#pragma unroll
      for (int i = 0; i < MAXV; ++i) {
        const int c = LN_COL(i);
        if (c < nv) {
          const float4 x = make_float4(v[i].x * sc, v[i].y * sc, v[i].z * sc, v[i].w * sc);
          const __half2 a0 = __floats2half2_rn(x.x, x.y), a1 = __floats2half2_rn(x.z, x.w);
          const float2 f0 = __half22float2(a0), f1 = __half22float2(a1);
          const __half2 b0 = __floats2half2_rn(x.x - f0.x, x.y - f0.y), b1 = __floats2half2_rn(x.z - f1.x, x.w - f1.y);
          *reinterpret_cast<uint2 *>(p1 + 4 * c) = make_uint2(*reinterpret_cast<const uint32_t *>(&a0), *reinterpret_cast<const uint32_t *>(&a1));
          *reinterpret_cast<uint2 *>(p2 + 4 * c) = make_uint2(*reinterpret_cast<const uint32_t *>(&b0), *reinterpret_cast<const uint32_t *>(&b1));
        }
      }
      for (int c = d + lane; c < Kp; c += 32) { p1[c] = __float2half(0.0f); p2[c] = __float2half(0.0f); }
      continue;
    }
#pragma unroll
    for (int i = 0; i < MAXV; i += 2) {
      const int c = LN_COL(i);   // even float4 column; c + 1 is register i + 1
      float4 o[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (c + h < nv) {
          if (sum_out) reinterpret_cast<float4 *>(sum_out + (int64_t)row * d)[c + h] = v[i + h];
          const float4 g = __ldg(reinterpret_cast<const float4 *>(gamma) + c + h);
          const float4 be = __ldg(reinterpret_cast<const float4 *>(beta) + c + h);
          o[h].x = (v[i + h].x - mean) * rstd * g.x + be.x;
          o[h].y = (v[i + h].y - mean) * rstd * g.y + be.y;
          o[h].z = (v[i + h].z - mean) * rstd * g.z + be.z;
          o[h].w = (v[i + h].w - mean) * rstd * g.w + be.w;
          reinterpret_cast<float4 *>(y + (int64_t)row * d)[c + h] = o[h];
          if (y_hi) reinterpret_cast<float4 *>(y_hi + (int64_t)row * Kp)[c + h] = o[h];
        }
      }
      if (y_lo) {  // operand pair for the next GEMM; y itself serves as `hi` when no K padding is needed (y_hi == NULL)
        if (c + 1 < nv) corr_store8(y_lo + (int64_t)row * Kp, 4 * c, o[0], o[1], 0);
        else if (c < nv) corr_store4(y_lo + (int64_t)row * Kp, 4 * c, o[0], 0);
      }
    }
#undef LN_COL
    if (y_lo)
      for (int c = d + lane; c < Kp; c += 32) {
        if (y_hi) y_hi[(int64_t)row * Kp + c] = 0.0f;
        corr_store1(y_lo + (int64_t)row * Kp, c, 0.0f, 0);
      }
  }
}

// GELU(erf) + hi/lo split: src [rows, cols] (row stride ld) -> hi/lo [rows, Kp]
__global__ void __launch_bounds__(256) gelu_split_kernel(const float *__restrict__ src, int64_t ld, int rows, int cols,
                                                         int Kp, float *__restrict__ act, float *__restrict__ hi,
                                                         float *__restrict__ lo) {
  const int64_t total = (int64_t)rows * Kp;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(idx % Kp);
    const int64_t r = idx / Kp;
    const float v = (k < cols) ? gelu_erf(__ldg(src + r * ld + k)) : 0.0f;
    if (act && k < cols) act[r * cols + k] = v;
    hi[idx] = v;
    corr_store1(lo + r * Kp, k, v, 0);
  }
}

// the same, 8 consecutive columns per thread (16-byte loads and stores); needs cols % 8 == 0 and 16-byte aligned rows
__global__ void __launch_bounds__(256) gelu_split_v8_kernel(const float *__restrict__ src, int64_t ld, int rows, int cols,
                                                            int Kp, float *__restrict__ act, float *__restrict__ hi,
                                                            float *__restrict__ lo) {
  const int k8n = Kp >> 3;
  const int64_t total = (int64_t)rows * k8n;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(idx % k8n) << 3;
    const int64_t r = idx / k8n;
    float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
    if (k < cols) {
      v0 = __ldg(reinterpret_cast<const float4 *>(src + r * ld + k));
      v1 = __ldg(reinterpret_cast<const float4 *>(src + r * ld + k) + 1);
      v0 = make_float4(gelu_erf(v0.x), gelu_erf(v0.y), gelu_erf(v0.z), gelu_erf(v0.w));
      v1 = make_float4(gelu_erf(v1.x), gelu_erf(v1.y), gelu_erf(v1.z), gelu_erf(v1.w));
      if (act) {
        reinterpret_cast<float4 *>(act + r * cols + k)[0] = v0;
        reinterpret_cast<float4 *>(act + r * cols + k)[1] = v1;
      }
    }
    reinterpret_cast<float4 *>(hi + r * Kp + k)[0] = v0;
    reinterpret_cast<float4 *>(hi + r * Kp + k)[1] = v1;
    corr_store8(lo + r * Kp, k, v0, v1, 0);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Banded attention, forward.  One CTA per (32-query block, head, episode); key/value tiles of 64 rows are
// staged in shared memory and ONLY the tiles intersecting [q0 - w, q0 + 32 + w) x [0, len_b) are read
// (HF's sliding chunks compute 2w x 2w blocks and mask half of them away).  Running-max softmax in fp32
// (HF: softmax in fp32, modeling_longformer.py:573), exact zeros for padded queries (:578).
//   phases 1 + 2  S = Q K^T and the running softmax, warp-local: warp = 4 queries x the 64 keys of the tile (thread =
//             4 queries x 2 keys, float4 along the head dimension, FFMA2); row max / exp / sum by shuffles, the four rows
//             interleaved; running statistics in registers; P and the rescale factors go to shared memory
//   phase 3   O = alpha O + P V   warp = 4 float4 head columns, thread = 4 queries x 1 float4 column (FFMA2); heads wider
//             than 128 (NCW = 2): thread = 4 queries x the float4 columns cg and cg + 32, sharing the P loads
// Three block-wide barriers per tile; K / V tiles by cp.async.
// Shared rows are padded to a stride = 4 (mod 8) words so that 8 consecutive rows read as float4 hit
// 8 distinct bank groups.
// ---------------------------------------------------------------------------------------------------------
constexpr int BA_BQ = 32, BA_TK = 64, BA_THREADS = 256, BA_PS = BA_TK + 4;

__host__ __device__ inline int ba_row_stride(int hd) { return (hd % 8 == 0) ? hd + 4 : hd; }
static size_t ba_smem_bytes(int hd) {
  return sizeof(float) * ((size_t)(BA_BQ + 2 * BA_TK) * ba_row_stride(hd) + BA_BQ * BA_PS + 3 * BA_BQ);
}

// DROP: dropout on the probabilities (training): the weights of P V are p * keep / (1 - p_drop), the softmax denominator
// and the saved log-sum-exp stay those of the undropped probabilities (attn_keep_scale, common.cuh).
// NCW: float4 head columns per phase-3 thread, 1 for hd <= 128, 2 for 128 < hd <= 256.
template <bool DROP, int NCW>
__global__ void __launch_bounds__(BA_THREADS, 2)
    band_attn_fwd_kernel(const float *__restrict__ qkv, int64_t ld, const int32_t *__restrict__ lengths,
                         const int32_t *__restrict__ offsets, int S, int nheads, int hd, int w,
                         float *__restrict__ out, float *__restrict__ out_hi, float *__restrict__ out_lo, int Kp,
                         float *__restrict__ lse, uint32_t p24, float inv_keep, uint64_t seed) {
  extern __shared__ __align__(16) float sm[];
  const int RS = ba_row_stride(hd);
  float *Qs = sm;
  float *Ks = Qs + BA_BQ * RS;
  float *Vs = Ks + BA_TK * RS;
  float *Ps = Vs + BA_TK * RS;
  float *m_s = Ps + BA_BQ * BA_PS;
  float *l_s = m_s + BA_BQ;
  float *al_s = l_s + BA_BQ;

  const int b = blockIdx.z, head = blockIdx.y, q0 = blockIdx.x * BA_BQ;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int d = nheads * hd, nv = hd >> 2;
  const int len = min(max(lengths[b], 0), S);
  // ragged layout (offsets != NULL): episode b owns rows offsets[b] .. offsets[b] + len - 1 and nothing beyond
  const int64_t row0 = offsets ? (int64_t)offsets[b] : (int64_t)b * S;
  const int Sq = offsets ? len : S;  // rows of this episode that exist in memory
  // Phase-3 lane mapping: a warp-wide 16-byte shared-memory load touches 128 contiguous-bank bytes (one wavefront):
  // the 8 lane groups (lane >> 2) take 8 consecutive P rows, the 4 lanes of a group 4 consecutive 16-byte V columns;
  // warp = 4 float4 head columns, thread = 4 queries (qgrp + 8r) x 1 float4 column.
  const int qgrp = lane >> 2;
  const int cg = 4 * warp + (lane & 3);   // phase 3 / output: my float4 column of the head (and cg + 32 .. when NCW > 1)
  const bool pv_thread = cg < nv;
  // column of chunk c; a thread whose cg + 32 c lies past the head computes the last column again and does not store it
  auto col = [&](int c) { return c == 0 ? cg : min(cg + 32 * c, nv - 1); };
  auto col_ok = [&](int c) { return c == 0 || cg + 32 * c < nv; };

  if (q0 >= len) {  // whole block is padding: exact zeros
    if (pv_thread) {
#pragma unroll
      for (int c = 0; c < NCW; ++c) {
        if (!col_ok(c)) continue;
        const int cc = col(c);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int i = q0 + qgrp + 8 * r;
          if (i < Sq) {
            const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
            if (out) reinterpret_cast<float4 *>(out + (row0 + i) * d + head * hd)[cc] = z;
            if (out_hi) {
              reinterpret_cast<float4 *>(out_hi + (row0 + i) * Kp + head * hd)[cc] = z;
              corr_store4(out_lo + (row0 + i) * Kp, head * hd + 4 * cc, z, 0);
            }
          }
        }
      }
    }
    if (lse && tid < BA_BQ && q0 + tid < S) lse[((int64_t)b * nheads + head) * S + q0 + tid] = 0.0f;
    return;
  }

  const float scale = sqrtf((float)hd);
  for (int idx = tid; idx < BA_BQ * nv; idx += BA_THREADS) {
    const int r = idx / nv, c = idx % nv;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q0 + r < Sq) {
      v = __ldg(reinterpret_cast<const float4 *>(qkv + (row0 + q0 + r) * ld + head * hd) + c);
      v.x /= scale; v.y /= scale; v.z /= scale; v.w /= scale;  // query_vectors /= sqrt(head_dim) (HF :513)
    }
    reinterpret_cast<float4 *>(Qs + r * RS)[c] = v;
  }
  float m_run[4], l_run[4];   // running max / sum of my warp's 4 query rows (same value in every lane)
#pragma unroll
  for (int a = 0; a < 4; ++a) { m_run[a] = -INFINITY; l_run[a] = 0.0f; }

  float2 o2[NCW][4][2];   // per float4 head column: 4 queries x (columns 0-1, columns 2-3)
#pragma unroll
  for (int c = 0; c < NCW; ++c)
#pragma unroll
    for (int r = 0; r < 4; ++r) o2[c][r][0] = o2[c][r][1] = make_float2(0.0f, 0.0f);

  const int kbeg = max(0, q0 - w), kend = min(len, q0 + BA_BQ + w);

  // K / V tiles arrive by cp.async (16-byte LDGSTS, zero-filled beyond kend) and overlap the arithmetic without extra
  // buffers: V_t is requested at the top of tile t and only awaited before phase 3; K_{t+1} is requested as soon as
  // phase 1 of tile t has released the K buffer.
  // (row, 16-byte column) of my first piece of a tile and the step to my next one: no division in the loops
  const int r_first = tid / nv, c_first = tid % nv, r_step = BA_THREADS / nv, c_step = BA_THREADS % nv;
  auto request_tile = [&](float *dst, int k0, int which) {
    const float *gbase = qkv + (row0 + k0) * ld + head * hd + which * d;
    int r = r_first, c = c_first;
    while (r < BA_TK) {
      const bool valid = k0 + r < kend;
      const float *src = valid ? gbase + (int64_t)r * ld + 4 * c : qkv;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst + r * RS + 4 * c)),
                   "l"(src), "r"(valid ? 16 : 0)
                   : "memory");
      r += r_step;
      c += c_step;
      if (c >= nv) { c -= nv; ++r; }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  request_tile(Ks, kbeg, 1);

  for (int k0 = kbeg; k0 < kend; k0 += BA_TK) {
    request_tile(Vs, k0, 2);
    asm volatile("cp.async.wait_group 1;" ::: "memory");  // K_t has landed (V_t may still be in flight)
    __syncthreads();
    // ---- phases 1 + 2: scores and running softmax, warp-local (warp = 4 queries x the 64 keys of the tile) -------
    {
      // packed fp32 FMAs (FFMA2): Blackwell issues scalar FFMA at half rate.  Pairs run over consecutive head
      // dimensions: (even-index sum, odd-index sum), added at the end.
      float2 acc2[4][2];
#pragma unroll
      for (int a = 0; a < 4; ++a) acc2[a][0] = acc2[a][1] = make_float2(0.0f, 0.0f);
      const float4 *qp = reinterpret_cast<const float4 *>(Qs + 4 * warp * RS);
      const float4 *kp0 = reinterpret_cast<const float4 *>(Ks + lane * RS);
      const float4 *kp1 = reinterpret_cast<const float4 *>(Ks + (lane + 32) * RS);
      const int qstep = RS / 4;   // next query row, in float4
      for (int c = 0; c < nv; ++c) {
        const float4 ka = kp0[c], kb = kp1[c];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          const float4 x = qp[a * qstep + c];   // same address in every lane: broadcast
          const float2 xl = make_float2(x.x, x.y), xh = make_float2(x.z, x.w);
          acc2[a][0] = __ffma2_rn(xh, make_float2(ka.z, ka.w), __ffma2_rn(xl, make_float2(ka.x, ka.y), acc2[a][0]));
          acc2[a][1] = __ffma2_rn(xh, make_float2(kb.z, kb.w), __ffma2_rn(xl, make_float2(kb.x, kb.y), acc2[a][1]));
        }
      }
      float sc[4][2], mx[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int i = q0 + 4 * warp + a;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int kj = k0 + lane + 32 * j;
          const bool ok = (i < len) && (kj < kend) && (kj >= i - w) && (kj <= i + w);
          sc[a][j] = ok ? acc2[a][j].x + acc2[a][j].y : -INFINITY;
        }
        mx[a] = fmaxf(sc[a][0], sc[a][1]);
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1)
#pragma unroll
        for (int a = 0; a < 4; ++a) mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], off));
      float ps[4], alpha[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const float m_new = fmaxf(m_run[a], mx[a]);
        const float m_use = (m_new == -INFINITY) ? 0.0f : m_new;
        const float p0 = expf(sc[a][0] - m_use), p1 = expf(sc[a][1] - m_use);
        float pv0 = p0, pv1 = p1;
        if (DROP) {
          const uint32_t bh = (uint32_t)(b * nheads + head), i = (uint32_t)(q0 + 4 * warp + a);
          pv0 *= attn_keep_scale(seed, bh, i, (uint32_t)(k0 + lane), p24, inv_keep);
          pv1 *= attn_keep_scale(seed, bh, i, (uint32_t)(k0 + lane + 32), p24, inv_keep);
        }
        Ps[(4 * warp + a) * BA_PS + lane] = pv0;
        Ps[(4 * warp + a) * BA_PS + lane + 32] = pv1;
        ps[a] = p0 + p1;
        alpha[a] = expf(m_run[a] - m_use);
        m_run[a] = m_new;
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1)
#pragma unroll
        for (int a = 0; a < 4; ++a) ps[a] += __shfl_xor_sync(0xffffffffu, ps[a], off);
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        l_run[a] = l_run[a] * alpha[a] + ps[a];
        if (lane == 0) al_s[4 * warp + a] = alpha[a];
      }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");  // my pieces of V_t have landed
    __syncthreads();                                       // P, alpha and V_t visible to all; the K buffer is free
    if (k0 + BA_TK < kend) request_tile(Ks, k0 + BA_TK, 1);
    // ---- phase 3: O = alpha O + P V ----------------------------------------------------------------------
    if (pv_thread) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const float al = al_s[qgrp + 8 * r];
#pragma unroll
        for (int c = 0; c < NCW; ++c) {
          o2[c][r][0] = __fmul2_rn(o2[c][r][0], make_float2(al, al));
          o2[c][r][1] = __fmul2_rn(o2[c][r][1], make_float2(al, al));
        }
      }
#pragma unroll 4
      for (int k4 = 0; k4 < BA_TK / 4; ++k4) {
        float4 p[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) p[r] = reinterpret_cast<const float4 *>(Ps + (qgrp + 8 * r) * BA_PS)[k4];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
          for (int c = 0; c < NCW; ++c) {
            const float4 vv = reinterpret_cast<const float4 *>(Vs + (4 * k4 + kk) * RS)[col(c)];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              const float pk = kk == 0 ? p[r].x : kk == 1 ? p[r].y : kk == 2 ? p[r].z : p[r].w;
              const float2 pk2 = make_float2(pk, pk);
              o2[c][r][0] = __ffma2_rn(pk2, make_float2(vv.x, vv.y), o2[c][r][0]);
              o2[c][r][1] = __ffma2_rn(pk2, make_float2(vv.z, vv.w), o2[c][r][1]);
            }
          }
        }
      }
    }
    __syncthreads();
  }
  if (lane == 0) {
#pragma unroll
    for (int a = 0; a < 4; ++a) { m_s[4 * warp + a] = m_run[a]; l_s[4 * warp + a] = l_run[a]; }
  }
  __syncthreads();

  if (pv_thread) {
#pragma unroll
    for (int c = 0; c < NCW; ++c) {
      if (!col_ok(c)) continue;
      const int cc = col(c);
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int i = q0 + qgrp + 8 * r;
        if (i >= Sq) continue;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < len) {
          const float inv = 1.0f / l_s[qgrp + 8 * r];
          v = make_float4(o2[c][r][0].x * inv, o2[c][r][0].y * inv, o2[c][r][1].x * inv, o2[c][r][1].y * inv);
        }
        if (out) reinterpret_cast<float4 *>(out + (row0 + i) * d + head * hd)[cc] = v;
        if (out_hi) {
          reinterpret_cast<float4 *>(out_hi + (row0 + i) * Kp + head * hd)[cc] = v;
          corr_store4(out_lo + (row0 + i) * Kp, head * hd + 4 * cc, v, 0);
        }
      }
    }
  }
  if (lse && tid < BA_BQ && q0 + tid < S)
    lse[((int64_t)b * nheads + head) * S + q0 + tid] = (q0 + tid < len) ? m_s[tid] + logf(l_s[tid]) : 0.0f;
}

// ---------------------------------------------------------------------------------------------------------
// Banded attention, forward, on the tensor cores: warp-level mma.sync m16n8k8 TF32 with 3xTF32 error compensation
// (x = hi + lo, hi = the 19 bits the tensor core keeps, products hi*hi + hi*lo + lo*hi: fp32-grade scores and outputs).
// One CTA = 64 queries of one head (4 warps x 16 rows); K/V tiles of 64 keys in shared memory; every warp only
// multiplies the 8-key column tiles that intersect ITS 16-row band, so small windows do proportionally less work.
// Q fragments stay in registers for the whole CTA; S never leaves registers: the accumulator fragment of S
// (rows g, g+8; keys 2t, 2t+1) is re-used directly as the A fragment of P V by pairing MMA k-index t with key 2t and
// t+4 with key 2t+1 on the V side (no shuffles, no shared-memory round trip).  Shared rows have stride hd + 4 words
// (= 4 mod 8), which makes both the K-fragment reads (8 keys x 4 k) and the V-fragment reads (4 key pairs x 8
// columns) bank-conflict free.
// ---------------------------------------------------------------------------------------------------------
constexpr int BM_BQ = 64, BM_TK = 64, BM_THREADS = 128;

__device__ __forceinline__ void mma_tf32_16x8x8(float (&d)[4], const uint32_t a0, const uint32_t a1, const uint32_t a2,
                                                const uint32_t a3, const uint32_t b0, const uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t tf32_hi_bits(float x) { return __float_as_uint(x) & 0xFFFFE000u; }
__device__ __forceinline__ uint32_t tf32_lo_bits(float x, uint32_t hi) { return __float_as_uint(x - __uint_as_float(hi)); }

template <int NHD>  // head dim / 8
__global__ void __launch_bounds__(BM_THREADS, 2)
    band_attn_fwd_mma_kernel(const float *__restrict__ qkv, int64_t ld, const int32_t *__restrict__ lengths,
                             const int32_t *__restrict__ offsets, int S, int nheads, int w, float *__restrict__ out,
                             float *__restrict__ out_hi, float *__restrict__ out_lo, int Kp, float *__restrict__ lse) {
  constexpr int HD = NHD * 8, RS = HD + 4, NV = HD / 4;
  extern __shared__ __align__(16) float sm[];
  float *Ks = sm;                 // [64][RS]  (first holds the scaled Q tile)
  float *Vs = Ks + BM_TK * RS;    // [64][RS]

  const int b = blockIdx.z, head = blockIdx.y, q0 = blockIdx.x * BM_BQ;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int d = nheads * HD;
  const int len = min(max(lengths[b], 0), S);
  // ragged layout (offsets != NULL): episode b owns rows offsets[b] .. offsets[b] + len - 1 and nothing beyond
  const int64_t row0 = offsets ? (int64_t)offsets[b] : (int64_t)b * S;
  const int Sq = offsets ? len : S;  // rows of this episode that exist in memory
  const int r0 = q0 + 16 * warp;             // first query row of this warp
  const int ia = r0 + g, ib = r0 + g + 8;    // the two rows this thread holds

  if (q0 >= len) {  // whole block is padding: exact zeros
    for (int idx = tid; idx < BM_BQ * NV; idx += BM_THREADS) {
      const int r = idx / NV, c = idx % NV;
      if (q0 + r < Sq) {
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        if (out) reinterpret_cast<float4 *>(out + (row0 + q0 + r) * d + head * HD)[c] = z;
        if (out_hi) {
          reinterpret_cast<float4 *>(out_hi + (row0 + q0 + r) * Kp + head * HD)[c] = z;
          corr_store4(out_lo + (row0 + q0 + r) * Kp, head * HD + 4 * c, z, 0);
        }
      }
    }
    if (lse && tid < BM_BQ && q0 + tid < S) lse[((int64_t)b * nheads + head) * S + q0 + tid] = 0.0f;
    return;
  }

  // ---- Q tile -> shared (scaled as HF does, :513) -> A fragments in registers ------------------------------------
  const float scale = sqrtf((float)HD);
  for (int idx = tid; idx < BM_BQ * NV; idx += BM_THREADS) {
    const int r = idx / NV, c = idx % NV;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q0 + r < Sq) {
      v = __ldg(reinterpret_cast<const float4 *>(qkv + (row0 + q0 + r) * ld + head * HD) + c);
      v.x /= scale; v.y /= scale; v.z /= scale; v.w /= scale;
    }
    reinterpret_cast<float4 *>(Ks + r * RS)[c] = v;
  }
  __syncthreads();
  float aq[NHD][4];
#pragma unroll
  for (int ks = 0; ks < NHD; ++ks) {
    const float *qa = Ks + (16 * warp + g) * RS + 8 * ks + t;
    aq[ks][0] = qa[0]; aq[ks][1] = qa[8 * RS]; aq[ks][2] = qa[4]; aq[ks][3] = qa[8 * RS + 4];
  }
  __syncthreads();

  float oacc[NHD][4];
#pragma unroll
  for (int n = 0; n < NHD; ++n) { oacc[n][0] = oacc[n][1] = oacc[n][2] = oacc[n][3] = 0.0f; }
  float m_a = -INFINITY, m_b = -INFINITY, l_a = 0.0f, l_b = 0.0f;

  const int kbeg = max(0, q0 - w), kend = min(len, q0 + BM_BQ + w);
  for (int k0 = kbeg; k0 < kend; k0 += BM_TK) {
    for (int idx = tid; idx < BM_TK * NV; idx += BM_THREADS) {
      const int r = idx / NV, c = idx % NV;
      float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
      if (k0 + r < kend) {
        const float *base = qkv + (row0 + k0 + r) * ld + head * HD;
        kv = __ldg(reinterpret_cast<const float4 *>(base + d) + c);
        vv = __ldg(reinterpret_cast<const float4 *>(base + 2 * d) + c);
      }
      reinterpret_cast<float4 *>(Ks + r * RS)[c] = kv;
      reinterpret_cast<float4 *>(Vs + r * RS)[c] = vv;
    }
    __syncthreads();
    // 8-key column tiles of this K tile that intersect the band of my 16 rows (warp-uniform)
    int jlo = (r0 - w - k0) >> 3, jhi = (r0 + 15 + w - k0) >> 3;
    jlo = max(jlo, 0);
    jhi = min(jhi, min(BM_TK / 8 - 1, (kend - 1 - k0) >> 3));
    if (r0 < len && jlo <= jhi) {
      // ---- S = Q K^T on the active column tiles ------------------------------------------------------------------
      float sacc[BM_TK / 8][4];
#pragma unroll
      for (int j = 0; j < BM_TK / 8; ++j) { sacc[j][0] = sacc[j][1] = sacc[j][2] = sacc[j][3] = 0.0f; }
#pragma unroll
      for (int ks = 0; ks < NHD; ++ks) {
        const uint32_t h0 = tf32_hi_bits(aq[ks][0]), h1 = tf32_hi_bits(aq[ks][1]);
        const uint32_t h2 = tf32_hi_bits(aq[ks][2]), h3 = tf32_hi_bits(aq[ks][3]);
        const uint32_t l0 = tf32_lo_bits(aq[ks][0], h0), l1 = tf32_lo_bits(aq[ks][1], h1);
        const uint32_t l2 = tf32_lo_bits(aq[ks][2], h2), l3 = tf32_lo_bits(aq[ks][3], h3);
#pragma unroll
        for (int j = 0; j < BM_TK / 8; ++j) {
          if (j >= jlo && j <= jhi) {
            const float *kp = Ks + (8 * j + g) * RS + 8 * ks + t;
            const float kb0 = kp[0], kb1 = kp[4];
            const uint32_t bh0 = tf32_hi_bits(kb0), bh1 = tf32_hi_bits(kb1);
            const uint32_t bl0 = tf32_lo_bits(kb0, bh0), bl1 = tf32_lo_bits(kb1, bh1);
            mma_tf32_16x8x8(sacc[j], h0, h1, h2, h3, bh0, bh1);
            mma_tf32_16x8x8(sacc[j], h0, h1, h2, h3, bl0, bl1);
            mma_tf32_16x8x8(sacc[j], l0, l1, l2, l3, bh0, bh1);
          }
        }
      }
      // ---- band / length mask, running softmax (rows ia and ib) ---------------------------------------------------
      float mx_a = -INFINITY, mx_b = -INFINITY;
#pragma unroll
      for (int j = 0; j < BM_TK / 8; ++j) {
        const bool act = (j >= jlo && j <= jhi);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const int key = k0 + 8 * j + 2 * t + c;
          const bool oka = act && ia < len && key < kend && key >= ia - w && key <= ia + w;
          const bool okb = act && ib < len && key < kend && key >= ib - w && key <= ib + w;
          sacc[j][c] = oka ? sacc[j][c] : -INFINITY;
          sacc[j][2 + c] = okb ? sacc[j][2 + c] : -INFINITY;
          mx_a = fmaxf(mx_a, sacc[j][c]);
          mx_b = fmaxf(mx_b, sacc[j][2 + c]);
        }
      }
      mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 1)); mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 2));
      mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 1)); mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 2));
      const float mn_a = fmaxf(m_a, mx_a), mn_b = fmaxf(m_b, mx_b);
      const float mu_a = (mn_a == -INFINITY) ? 0.0f : mn_a, mu_b = (mn_b == -INFINITY) ? 0.0f : mn_b;
      const float al_a = expf(m_a - mu_a), al_b = expf(m_b - mu_b);
      m_a = mn_a; m_b = mn_b;
      float ps_a = 0.0f, ps_b = 0.0f;
#pragma unroll
      for (int j = 0; j < BM_TK / 8; ++j) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          sacc[j][c] = expf(sacc[j][c] - mu_a);
          sacc[j][2 + c] = expf(sacc[j][2 + c] - mu_b);
          ps_a += sacc[j][c];
          ps_b += sacc[j][2 + c];
        }
      }
      l_a = l_a * al_a + ps_a;   // per-thread partial row sums; reduced over the quad at the end
      l_b = l_b * al_b + ps_b;
#pragma unroll
      for (int n = 0; n < NHD; ++n) { oacc[n][0] *= al_a; oacc[n][1] *= al_a; oacc[n][2] *= al_b; oacc[n][3] *= al_b; }
      // ---- O += P V: the S accumulator fragment is the A fragment (k-index t <-> key 2t, t+4 <-> key 2t+1) ----------
#pragma unroll
      for (int j = 0; j < BM_TK / 8; ++j) {
        if (j >= jlo && j <= jhi) {
          const uint32_t h0 = tf32_hi_bits(sacc[j][0]), h1 = tf32_hi_bits(sacc[j][2]);
          const uint32_t h2 = tf32_hi_bits(sacc[j][1]), h3 = tf32_hi_bits(sacc[j][3]);
          const uint32_t l0 = tf32_lo_bits(sacc[j][0], h0), l1 = tf32_lo_bits(sacc[j][2], h1);
          const uint32_t l2 = tf32_lo_bits(sacc[j][1], h2), l3 = tf32_lo_bits(sacc[j][3], h3);
          const float *vp = Vs + (8 * j + 2 * t) * RS + g;
#pragma unroll
          for (int n = 0; n < NHD; ++n) {
            const float vb0 = vp[8 * n], vb1 = vp[RS + 8 * n];
            const uint32_t bh0 = tf32_hi_bits(vb0), bh1 = tf32_hi_bits(vb1);
            const uint32_t bl0 = tf32_lo_bits(vb0, bh0), bl1 = tf32_lo_bits(vb1, bh1);
            mma_tf32_16x8x8(oacc[n], h0, h1, h2, h3, bh0, bh1);
            mma_tf32_16x8x8(oacc[n], h0, h1, h2, h3, bl0, bl1);
            mma_tf32_16x8x8(oacc[n], l0, l1, l2, l3, bh0, bh1);
          }
        }
      }
    }
    __syncthreads();
  }

  l_a += __shfl_xor_sync(0xffffffffu, l_a, 1); l_a += __shfl_xor_sync(0xffffffffu, l_a, 2);
  l_b += __shfl_xor_sync(0xffffffffu, l_b, 1); l_b += __shfl_xor_sync(0xffffffffu, l_b, 2);
  const float inv_a = (ia < len) ? 1.0f / l_a : 0.0f, inv_b = (ib < len) ? 1.0f / l_b : 0.0f;
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int i = half ? ib : ia;
    if (i >= Sq) continue;
    const float inv = half ? inv_b : inv_a;
#pragma unroll
    for (int n = 0; n < NHD; ++n) {
      const float2 v = make_float2(oacc[n][2 * half] * inv, oacc[n][2 * half + 1] * inv);
      const int col = head * HD + 8 * n + 2 * t;
      if (out) *reinterpret_cast<float2 *>(out + (row0 + i) * d + col) = v;
      if (out_hi) {
        *reinterpret_cast<float2 *>(out_hi + (row0 + i) * Kp + col) = v;
        corr_store2(out_lo + (row0 + i) * Kp, col, v, 0);
      }
    }
    if (lse && t == 0)
      lse[((int64_t)b * nheads + head) * S + i] = (i < len) ? (half ? m_b + logf(l_b) : m_a + logf(l_a)) : 0.0f;
  }
}

template <int NHD>
static int launch_band_mma(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B, int S,
                           int nheads, int w, float *out, float *out_hi, float *out_lo, int Kp, float *lse, cudaStream_t st) {
  constexpr int HD = NHD * 8;
  const size_t smem = sizeof(float) * 2 * BM_TK * (HD + 4);
  MTS_PER_DEVICE(bool, attr_set);
  if (!attr_set) {
    MTS_CUDA(cudaFuncSetAttribute(band_attn_fwd_mma_kernel<NHD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  const dim3 grid((S + BM_BQ - 1) / BM_BQ, nheads, B);
  band_attn_fwd_mma_kernel<NHD><<<grid, BM_THREADS, smem, st>>>(qkv, ld, lengths, offsets, S, nheads, w, out, out_hi, out_lo,
                                                                Kp, lse);
  MTS_LAUNCH_CHECK();
  return 0;
}

static unsigned ew_grid(int64_t total) {
  int64_t g = (total + 255) / 256;
  const int64_t cap = (int64_t)kNumSMs * 16;
  return (unsigned)(g < cap ? (g > 0 ? g : 1) : cap);
}

}  // namespace mts

using namespace mts;

static int ln_args_ok(const char *who, int M, int d, const float *y_hi, const float *y_lo, int Kp) {
  (void)who;
  if (M <= 0 || d <= 0) { set_error("layer norm: empty shape"); return MTS_E_BADARG; }
  if (d % 4 != 0 || d > 128 * LN_MAXV) { set_error("layer norm: width must be a multiple of 4 and <= 2048"); return MTS_E_UNSUPPORTED; }
  if (y_hi && !y_lo) { set_error("layer norm: hi without lo"); return MTS_E_BADARG; }
  if (y_lo && !y_hi && Kp != d) { set_error("layer norm: y can only stand in for hi when Kp == d"); return MTS_E_BADARG; }
  if (y_lo && (Kp % 32 != 0 || Kp < d)) { set_error("layer norm: Kp must be a multiple of 32 and >= d"); return MTS_E_BADARG; }
  return 0;
}

extern "C" int mts_embed_ln_fwd(const float *x, int64_t x_bstride, const float *pos, const float *typ,
                                const float *gamma, const float *beta, int B, int S, int d, float eps, float *y,
                                float *y_hi, float *y_lo, int Kp, float *sum_out, float *stats,
                                const int32_t *lengths, const int32_t *offsets, void *stream) {
  MTS_REQUIRE(x && pos && typ && gamma && beta && y, MTS_E_BADARG, "embed_ln_fwd: null pointer");
  MTS_REQUIRE(!offsets || lengths, MTS_E_BADARG, "embed_ln_fwd: ragged output needs the lengths");
  MTS_REQUIRE(B > 0 && S > 0, MTS_E_BADARG, "embed_ln_fwd: empty shape");
  int rc = ln_args_ok("embed_ln_fwd", B * S, d, y_hi, y_lo, Kp);
  if (rc) return rc;
  const int M = B * S;
  const unsigned grid = (unsigned)min((int64_t)(M + 7) / 8, (int64_t)kNumSMs * 8);
  if (d <= 1024)
    ln_fwd_kernel<0, 8><<<grid, 256, 0, (cudaStream_t)stream>>>(x, x_bstride, pos, typ, gamma, beta, M, S, d, eps, y, y_hi,
                                                                 y_lo, Kp, sum_out, stats, lengths, offsets);
  else
    ln_fwd_kernel<0, 16><<<grid, 256, 0, (cudaStream_t)stream>>>(x, x_bstride, pos, typ, gamma, beta, M, S, d, eps, y, y_hi,
                                                                  y_lo, Kp, sum_out, stats, lengths, offsets);
  MTS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mts_add_ln_fwd(const float *a, const float *res, const float *gamma, const float *beta, int M, int d,
                              float eps, float *y, float *y_hi, float *y_lo, int Kp, float *sum_out, float *stats,
                              void *stream) {
  MTS_REQUIRE(a && gamma && beta && y, MTS_E_BADARG, "add_ln_fwd: null pointer");  // res may be null: a = the sum
  int rc = ln_args_ok("add_ln_fwd", M, d, y_hi, y_lo, Kp);
  if (rc) return rc;
  const unsigned grid = (unsigned)min((int64_t)(M + 7) / 8, (int64_t)kNumSMs * 8);
  if (d <= 1024)
    ln_fwd_kernel<1, 8><<<grid, 256, 0, (cudaStream_t)stream>>>(a, 0, res, nullptr, gamma, beta, M, 0, d, eps, y, y_hi, y_lo,
                                                                 Kp, sum_out, stats, nullptr, nullptr);
  else
    ln_fwd_kernel<1, 16><<<grid, 256, 0, (cudaStream_t)stream>>>(a, 0, res, nullptr, gamma, beta, M, 0, d, eps, y, y_hi, y_lo,
                                                                  Kp, sum_out, stats, nullptr, nullptr);
  MTS_LAUNCH_CHECK();
  return 0;
}

// mts_embed_ln_fwd reading bf16 embeddings x (element stride x_bstride between episodes): y fp32 and its packed operand y_lo
// [rows, Kp] (side 0), the A operand of mts_gemm_bf16p / mts_gemm_bf16p_out16.  Everything after the load is mts_embed_ln_fwd's.
extern "C" int mts_embed_ln_fwd_bf16in(const void *x, int64_t x_bstride, const float *pos, const float *typ, const float *gamma,
                                       const float *beta, int B, int S, int d, float eps, float *y, float *y_lo, int Kp,
                                       const int32_t *lengths, const int32_t *offsets, void *stream) {
  MTS_REQUIRE(x && pos && typ && gamma && beta && y, MTS_E_BADARG, "embed_ln_fwd_bf16in: null pointer");
  MTS_REQUIRE(!offsets || lengths, MTS_E_BADARG, "embed_ln_fwd_bf16in: ragged output needs the lengths");
  MTS_REQUIRE(B > 0 && S > 0, MTS_E_BADARG, "embed_ln_fwd_bf16in: empty shape");
  MTS_REQUIRE(((uintptr_t)x & 7) == 0 && x_bstride % 4 == 0, MTS_E_BADARG, "embed_ln_fwd_bf16in: x must be 8-byte aligned, stride a multiple of 4");
  int rc = ln_args_ok("embed_ln_fwd_bf16in", B * S, d, nullptr, y_lo, Kp);
  if (rc) return rc;
  const int M = B * S;
  const float *xf = reinterpret_cast<const float *>(x);
  const unsigned grid = (unsigned)min((int64_t)(M + 7) / 8, (int64_t)kNumSMs * 8);
  if (d <= 1024)
    ln_fwd_kernel<2, 8><<<grid, 256, 0, (cudaStream_t)stream>>>(xf, x_bstride, pos, typ, gamma, beta, M, S, d, eps, y, nullptr, y_lo,
                                                                 Kp, nullptr, nullptr, lengths, offsets);
  else
    ln_fwd_kernel<2, 16><<<grid, 256, 0, (cudaStream_t)stream>>>(xf, x_bstride, pos, typ, gamma, beta, M, S, d, eps, y, nullptr, y_lo,
                                                                  Kp, nullptr, nullptr, lengths, offsets);
  MTS_LAUNCH_CHECK();
  return 0;
}

// The same two kernels writing the fp16-split operand of mts_gemm_f16x3 (pieces [rows][2][K64] fp16 + row_scale [rows]) next to y
extern "C" int mts_embed_ln_fwd_f16(const float *x, int64_t x_bstride, const float *pos, const float *typ, const float *gamma,
                                    const float *beta, int B, int S, int d, float eps, float *y, void *pieces, int K64,
                                    float *row_scale, const int32_t *lengths, const int32_t *offsets, void *stream) {
  MTS_REQUIRE(x && pos && typ && gamma && beta && y && pieces && row_scale, MTS_E_BADARG, "embed_ln_fwd_f16: null pointer");
  MTS_REQUIRE(!offsets || lengths, MTS_E_BADARG, "embed_ln_fwd_f16: ragged output needs the lengths");
  MTS_REQUIRE(B > 0 && S > 0 && d > 0 && d % 4 == 0 && d <= 1024, MTS_E_UNSUPPORTED, "embed_ln_fwd_f16: width must be a multiple of 4 and <= 1024");
  MTS_REQUIRE(K64 % 64 == 0 && K64 >= d, MTS_E_BADARG, "embed_ln_fwd_f16: K64 must be a multiple of 64 and >= d");
  const int M = B * S;
  const unsigned grid = (unsigned)min((int64_t)(M + 7) / 8, (int64_t)kNumSMs * 8);
  ln_fwd_kernel<0, 8, true><<<grid, 256, 0, (cudaStream_t)stream>>>(x, x_bstride, pos, typ, gamma, beta, M, S, d, eps, y, nullptr,
                                                                     reinterpret_cast<float *>(pieces), K64, nullptr, nullptr, lengths,
                                                                     offsets, row_scale);
  MTS_LAUNCH_CHECK();
  return 0;
}
extern "C" int mts_add_ln_fwd_f16(const float *a, const float *res, const float *gamma, const float *beta, int M, int d, float eps,
                                  float *y, void *pieces, int K64, float *row_scale, void *stream) {
  MTS_REQUIRE(a && gamma && beta && y && pieces && row_scale, MTS_E_BADARG, "add_ln_fwd_f16: null pointer");
  MTS_REQUIRE(M > 0 && d > 0 && d % 4 == 0 && d <= 1024, MTS_E_UNSUPPORTED, "add_ln_fwd_f16: width must be a multiple of 4 and <= 1024");
  MTS_REQUIRE(K64 % 64 == 0 && K64 >= d, MTS_E_BADARG, "add_ln_fwd_f16: K64 must be a multiple of 64 and >= d");
  const unsigned grid = (unsigned)min((int64_t)(M + 7) / 8, (int64_t)kNumSMs * 8);
  ln_fwd_kernel<1, 8, true><<<grid, 256, 0, (cudaStream_t)stream>>>(a, 0, res, nullptr, gamma, beta, M, 0, d, eps, y, nullptr,
                                                                     reinterpret_cast<float *>(pieces), K64, nullptr, nullptr, nullptr,
                                                                     nullptr, row_scale);
  MTS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mts_gelu_split(const float *src, int64_t ld, int rows, int cols, int Kp, float *act, float *hi,
                              float *lo, void *stream) {
  MTS_REQUIRE(src && hi && lo, MTS_E_BADARG, "gelu_split: null pointer");
  MTS_REQUIRE(rows > 0 && cols > 0 && Kp % 32 == 0 && Kp >= cols, MTS_E_BADARG, "gelu_split: bad shape");
  if (cols % 8 == 0 && ld % 4 == 0 && ((((uintptr_t)src | (uintptr_t)act | (uintptr_t)hi | (uintptr_t)lo) & 15) == 0))
    gelu_split_v8_kernel<<<ew_grid((int64_t)rows * (Kp / 8)), 256, 0, (cudaStream_t)stream>>>(src, ld, rows, cols, Kp, act, hi, lo);
  else
    gelu_split_kernel<<<ew_grid((int64_t)rows * Kp), 256, 0, (cudaStream_t)stream>>>(src, ld, rows, cols, Kp, act, hi, lo);
  MTS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mts_band_attn_fwd_mma(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B,
                                     int S, int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp,
                                     float *lse, void *stream) {
  MTS_REQUIRE(qkv && lengths && (out || out_hi), MTS_E_BADARG, "band_attn_fwd_mma: null pointer");
  MTS_REQUIRE((out_hi == nullptr) == (out_lo == nullptr), MTS_E_BADARG, "band_attn_fwd_mma: hi and lo go together");
  MTS_REQUIRE(B > 0 && S > 0 && nheads > 0 && hd > 0 && w >= 0, MTS_E_BADARG, "band_attn_fwd_mma: bad shape");
  MTS_REQUIRE(ld % 4 == 0 && ld >= 3 * nheads * hd, MTS_E_BADARG, "band_attn_fwd_mma: qkv row stride");
  MTS_REQUIRE(!out_hi || Kp == nheads * hd, MTS_E_UNSUPPORTED, "band_attn_fwd_mma: the split output needs Kp == model width");
  cudaStream_t st = (cudaStream_t)stream;
  switch (hd) {
    case 8: return launch_band_mma<1>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    case 16: return launch_band_mma<2>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    case 32: return launch_band_mma<4>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    case 64: return launch_band_mma<8>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    case 112: return launch_band_mma<14>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    case 128: return launch_band_mma<16>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    default: break;
  }
  set_error("band_attn_fwd_mma: head dim must be one of 8, 16, 32, 64, 112, 128");
  return MTS_E_UNSUPPORTED;
}

extern "C" int mts_band_attn_fwd(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B,
                                 int S, int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp,
                                 float *lse, void *stream) {
  // Default: the tcgen05 kernel (attn_tc.cu) for the head dims it is instantiated for; MTS_ATTN_IMPL=simt / mma select
  // the CUDA-core kernel below / the mma.sync kernel instead (second implementations for the tests).
  static const char *impl = getenv("MTS_ATTN_IMPL");
  if (impl && impl[0] == 'm' && (hd == 8 || hd == 16 || hd == 32 || hd == 64 || hd == 112 || hd == 128))
    return mts_band_attn_fwd_mma(qkv, ld, lengths, offsets, B, S, nheads, hd, w, out, out_hi, out_lo, Kp, lse, stream);
  if (!(impl && impl[0] == 's') && mts_band_attn_tc_supported(hd) && (!out_hi || Kp == nheads * hd))
    return mts_band_attn_fwd_tc(qkv, ld, lengths, offsets, B, S, nheads, hd, w, out, out_hi, out_lo, Kp, lse, stream);
  return mts_band_attn_fwd_simt(qkv, ld, lengths, offsets, B, S, nheads, hd, w, out, out_hi, out_lo, Kp, lse, stream);
}

template <int NCW>
static int band_attn_fwd_launch(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B, int S,
                                int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp, float *lse,
                                float p_drop, uint64_t seed, void *stream) {
  const size_t smem = ba_smem_bytes(hd);
  const dim3 grid((S + BA_BQ - 1) / BA_BQ, nheads, B);
  if (p_drop > 0.0f) {
    MTS_CUDA(cudaFuncSetAttribute(band_attn_fwd_kernel<true, NCW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    band_attn_fwd_kernel<true, NCW><<<grid, BA_THREADS, smem, (cudaStream_t)stream>>>(
        qkv, ld, lengths, offsets, S, nheads, hd, w, out, out_hi, out_lo, Kp, lse, attn_drop_p24(p_drop), 1.0f / (1.0f - p_drop), seed);
  } else {
    MTS_PER_DEVICE(size_t, smem_set);   // one per instantiation and device
    if (smem > smem_set) {
      MTS_CUDA(cudaFuncSetAttribute(band_attn_fwd_kernel<false, NCW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      smem_set = smem;
    }
    band_attn_fwd_kernel<false, NCW><<<grid, BA_THREADS, smem, (cudaStream_t)stream>>>(qkv, ld, lengths, offsets, S, nheads, hd, w,
                                                                                      out, out_hi, out_lo, Kp, lse, 0u, 1.0f, 0ull);
  }
  MTS_LAUNCH_CHECK();
  return 0;
}

static int band_attn_fwd_simt_impl(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B, int S,
                                   int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp, float *lse,
                                   float p_drop, uint64_t seed, void *stream) {
  MTS_REQUIRE(qkv && lengths && (out || out_hi), MTS_E_BADARG, "band_attn_fwd: null pointer");
  MTS_REQUIRE((out_hi == nullptr) == (out_lo == nullptr), MTS_E_BADARG, "band_attn_fwd: hi and lo go together");
  MTS_REQUIRE(B > 0 && S > 0 && nheads > 0 && hd > 0 && w >= 0, MTS_E_BADARG, "band_attn_fwd: bad shape");
  MTS_REQUIRE(hd % 4 == 0 && hd <= 256, MTS_E_UNSUPPORTED, "band_attn_fwd: head dim must be a multiple of 4 and <= 256");
  MTS_REQUIRE(ld % 4 == 0 && ld >= 3 * nheads * hd, MTS_E_BADARG, "band_attn_fwd: qkv row stride");
  MTS_REQUIRE(((uintptr_t)qkv & 15) == 0, MTS_E_BADARG, "band_attn_fwd: qkv must be 16-byte aligned");
  MTS_REQUIRE(!out_hi || (Kp % 32 == 0 && Kp >= nheads * hd), MTS_E_BADARG, "band_attn_fwd: Kp");
  MTS_REQUIRE(!out_hi || Kp == nheads * hd, MTS_E_UNSUPPORTED,
              "band_attn_fwd: the split output needs a model width that is a multiple of 32");
  MTS_REQUIRE(p_drop >= 0.0f && p_drop < 1.0f, MTS_E_BADARG, "band_attn_fwd: dropout probability must be in [0, 1)");
  MTS_REQUIRE(p_drop == 0.0f || S <= (1 << 20), MTS_E_UNSUPPORTED, "band_attn_fwd: dropout indices need S <= 2^20");
  if (hd > 128)
    return band_attn_fwd_launch<2>(qkv, ld, lengths, offsets, B, S, nheads, hd, w, out, out_hi, out_lo, Kp, lse, p_drop, seed, stream);
  return band_attn_fwd_launch<1>(qkv, ld, lengths, offsets, B, S, nheads, hd, w, out, out_hi, out_lo, Kp, lse, p_drop, seed, stream);
}

extern "C" int mts_band_attn_fwd_simt(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B,
                                      int S, int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp,
                                      float *lse, void *stream) {
  return band_attn_fwd_simt_impl(qkv, ld, lengths, offsets, B, S, nheads, hd, w, out, out_hi, out_lo, Kp, lse, 0.0f, 0ull, stream);
}

extern "C" int mts_band_attn_fwd_dropout(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B,
                                         int S, int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp,
                                         float *lse, float p_drop, uint64_t seed, void *stream) {
  return band_attn_fwd_simt_impl(qkv, ld, lengths, offsets, B, S, nheads, hd, w, out, out_hi, out_lo, Kp, lse, p_drop, seed, stream);
}
