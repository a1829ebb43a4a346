// Pyramidal windowed-attention encoder, backward kernels.  The reference has no hand-written backward: it is
// autograd through HF LongformerModel (models/CRF.py:574-594 -> loss.backward()).  These kernels produce the
// same gradients (SURVEY.md section 8a'):
//   LayerNorm       dx = rstd (g - mean(g) - xhat mean(g xhat)), g = dy gamma;  dgamma = sum dy xhat, dbeta = sum dy
//   GELU(erf)       dzp = dz (Phi(zp) + zp phi(zp))
//   banded softmax  dV = P^T dO, dP = dO V^T, dS = P (dP - rowsum(dO O)), dQ = dS K / sqrt(hd), dK = dS^T Q / sqrt(hd)
//                   restricted to |i-j| <= w, j < len_b, i < len_b, with P recomputed from the saved log-sum-exp
//   embeddings      dP[2 + t] = sum_b dpre[b, t], dE_type[0] = sum_{b,t} dpre[b, t]
// Every dX that feeds a tensor-core GEMM is also written as its operand pair (raw fp32 + bf16 correction, common.cuh)
// in the same pass.
#include "common.cuh"

namespace mts {

constexpr int LNB_MAXV = 16;

// one warp per row: dx (and its TF32 halves)
__global__ void __launch_bounds__(256) ln_bwd_dx_kernel(const float *__restrict__ dy, const float *__restrict__ pre,
                                                        const float *__restrict__ stats,
                                                        const float *__restrict__ gamma, int M, int d,
                                                        float *__restrict__ dx, float *__restrict__ dx_hi,
                                                        float *__restrict__ dx_lo, int Kp) {
  const int lane = threadIdx.x & 31;
  const int nv = d >> 2;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < M; row += warps) {
    const float mean = __ldg(stats + 2 * (int64_t)row), rstd = __ldg(stats + 2 * (int64_t)row + 1);
    float4 g[LNB_MAXV], xh[LNB_MAXV];
    float s1 = 0.0f, s2 = 0.0f;
#pragma unroll
    for (int i = 0; i < LNB_MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < nv) {
        const float4 a = __ldg(reinterpret_cast<const float4 *>(dy + (int64_t)row * d) + c);
        const float4 p = __ldg(reinterpret_cast<const float4 *>(pre + (int64_t)row * d) + c);
        const float4 w = __ldg(reinterpret_cast<const float4 *>(gamma) + c);
        g[i] = make_float4(a.x * w.x, a.y * w.y, a.z * w.z, a.w * w.w);
        xh[i] = make_float4((p.x - mean) * rstd, (p.y - mean) * rstd, (p.z - mean) * rstd, (p.w - mean) * rstd);
        s1 += (g[i].x + g[i].y) + (g[i].z + g[i].w);
        s2 += (g[i].x * xh[i].x + g[i].y * xh[i].y) + (g[i].z * xh[i].z + g[i].w * xh[i].w);
      }
    }
    const float m1 = warp_sum(s1) / (float)d, m2 = warp_sum(s2) / (float)d;
#pragma unroll
    for (int i = 0; i < LNB_MAXV; ++i) {
      const int c = lane + 32 * i;
      if (c < nv) {
        float4 o;
        o.x = rstd * (g[i].x - m1 - xh[i].x * m2);
        o.y = rstd * (g[i].y - m1 - xh[i].y * m2);
        o.z = rstd * (g[i].z - m1 - xh[i].z * m2);
        o.w = rstd * (g[i].w - m1 - xh[i].w * m2);
        reinterpret_cast<float4 *>(dx + (int64_t)row * d)[c] = o;
        if (dx_lo) {  // dx itself serves as `hi` when Kp == d (dx_hi == NULL)
          if (dx_hi) reinterpret_cast<float4 *>(dx_hi + (int64_t)row * Kp)[c] = o;
          corr_store4(dx_lo + (int64_t)row * Kp, 4 * c, o, 0);
        }
      }
    }
    if (dx_lo)
      for (int c = d + lane; c < Kp; c += 32) {
        if (dx_hi) dx_hi[(int64_t)row * Kp + c] = 0.0f;
        corr_store1(dx_lo + (int64_t)row * Kp, c, 0.0f, 0);
      }
  }
}

// column partial sums: CTA `blockIdx.x` owns a contiguous chunk of rows; thread = one float4 column
// partial [gridDim.x][2][d]  (dgamma part, dbeta part)
__global__ void __launch_bounds__(256) ln_bwd_param_kernel(const float *__restrict__ dy, const float *__restrict__ pre,
                                                           const float *__restrict__ stats, int M, int d,
                                                           int rows_per_cta, float *__restrict__ partial) {
  const int nv = d >> 2;
  const int r0 = blockIdx.x * rows_per_cta, r1 = min(M, r0 + rows_per_cta);
  for (int c = threadIdx.x; c < nv; c += blockDim.x) {
    float4 ag = make_float4(0.f, 0.f, 0.f, 0.f), ab = ag;
    for (int row = r0; row < r1; ++row) {
      const float mean = __ldg(stats + 2 * (int64_t)row), rstd = __ldg(stats + 2 * (int64_t)row + 1);
      const float4 a = __ldg(reinterpret_cast<const float4 *>(dy + (int64_t)row * d) + c);
      const float4 p = __ldg(reinterpret_cast<const float4 *>(pre + (int64_t)row * d) + c);
      ag.x = fmaf(a.x, (p.x - mean) * rstd, ag.x); ag.y = fmaf(a.y, (p.y - mean) * rstd, ag.y);
      ag.z = fmaf(a.z, (p.z - mean) * rstd, ag.z); ag.w = fmaf(a.w, (p.w - mean) * rstd, ag.w);
      ab.x += a.x; ab.y += a.y; ab.z += a.z; ab.w += a.w;
    }
    reinterpret_cast<float4 *>(partial + ((int64_t)blockIdx.x * 2 + 0) * d)[c] = ag;
    reinterpret_cast<float4 *>(partial + ((int64_t)blockIdx.x * 2 + 1) * d)[c] = ab;
  }
}

__global__ void __launch_bounds__(256) ln_bwd_param_final_kernel(const float *__restrict__ partial, int chunks, int d,
                                                                 float *__restrict__ dgamma, float *__restrict__ dbeta) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= 2 * d) return;
  float s = 0.0f;
  for (int k = 0; k < chunks; ++k) s += partial[(int64_t)k * 2 * d + c];
  if (c < d) dgamma[c] = s;
  else dbeta[c - d] = s;
}

// dzp = dz * d/dx GELU(zp), plus the TF32 halves of dzp
__global__ void __launch_bounds__(256) gelu_bwd_kernel(const float *__restrict__ dz, const float *__restrict__ zp,
                                                       int rows, int cols, int Kp, float *__restrict__ dzp,
                                                       float *__restrict__ hi, float *__restrict__ lo) {
  const int64_t total = (int64_t)rows * Kp;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(idx % Kp);
    const int64_t r = idx / Kp;
    float v = 0.0f;
    if (k < cols) {
      const float x = __ldg(zp + r * cols + k);
      const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
      const float pdf = 0.39894228040143267794f * expf(-0.5f * x * x);
      v = __ldg(dz + r * cols + k) * (cdf + x * pdf);
      dzp[r * cols + k] = v;
    }
    hi[idx] = v;
    corr_store1(lo + r * Kp, k, v, 0);
  }
}

// dpos[t, :] = sum_b dpre[b, t, :]
__global__ void __launch_bounds__(256) embed_bwd_kernel(const float *__restrict__ dpre, int B, int S, int d,
                                                        float *__restrict__ dpos, const int32_t *__restrict__ lengths,
                                                        const int32_t *__restrict__ offsets) {
  const int nv = d >> 2;
  const int64_t total = (int64_t)S * nv;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(idx % nv);
    const int64_t t = idx / nv;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int b = 0; b < B; ++b) {
      if (offsets && t >= lengths[b]) continue;  // ragged rows: position t of episode b exists only below its length
      const int64_t row = offsets ? (int64_t)offsets[b] + t : (int64_t)b * S + t;
      const float4 v = __ldg(reinterpret_cast<const float4 *>(dpre + row * d) + c);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    reinterpret_cast<float4 *>(dpos + t * d)[c] = acc;
  }
}

// ---------------------------------------------------------------------------------------------------------
// Banded attention backward.  Same tiling as the forward kernel (csrc/xfmr.cu): 32 "own" rows per CTA, 64-row
// tiles of the other side staged in shared memory, only tiles intersecting the band are read.
//   dq kernel : own rows = queries; loops key tiles;   writes dq and delta[i] = sum_c dO[i,c] O[i,c]
//   dkv kernel: own rows = keys;    loops query tiles; writes dk and dv (no atomics)
// Output mapping (the P dK / P^T dO products): thread = 4 own rows x 1 float4 head column (cg = tid % nv, needs nv <= 32); heads
// wider than 128 (NCW = 2): warp = 4 own rows, thread = the float4 columns cg and cg + 32 (cg = lane).
// ---------------------------------------------------------------------------------------------------------
constexpr int BB_OWN = 32, BB_TILE = 64, BB_THREADS = 256, BB_PS = BB_TILE + 4;

__host__ __device__ inline int bb_row_stride(int hd) { return (hd % 8 == 0) ? hd + 4 : hd; }

__device__ __forceinline__ float dot4(const float4 a, const float4 b, float acc) {
  return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, fmaf(a.w, b.w, acc))));
}

// DROP (both kernels): the forward pass weighted P V by p * m with m = keep / (1 - p_drop) (attn_keep_scale, regenerated here
// from the seed): dV = (P .* M)^T dO, dP = M .* (dO V^T), dS = P .* (dP - delta) with delta = rowsum(dO .* O) as before
// (sum_j P_ij dP_ij = dO_i . O_i holds with the dropped weights too).
// NCW (both kernels): float4 head columns per output thread, 1 for hd <= 128, 2 for 128 < hd <= 256.  The wide form keeps
// twice the accumulators and gets the whole register file: from hd 136 on, the shared memory of either kernel allows only one CTA
// per SM anyway.
template <bool DROP, int NCW>
__global__ void __launch_bounds__(BB_THREADS, NCW == 1 ? 2 : 1)
    band_attn_bwd_dq_kernel(const float *__restrict__ qkv, int64_t ld, const float *__restrict__ o,
                            const float *__restrict__ dO, const float *__restrict__ lse,
                            const int32_t *__restrict__ lengths, const int32_t *__restrict__ offsets, int S,
                            int nheads, int hd, int w, float *__restrict__ dqkv, float *__restrict__ delta,
                            uint32_t p24, float inv_keep, uint64_t seed) {
  extern __shared__ __align__(16) float sm[];
  const int RS = bb_row_stride(hd);
  float *Qs = sm;                       // [32][RS] scaled queries
  float *Gs = Qs + BB_OWN * RS;         // [32][RS] dO rows
  float *Ks = Gs + BB_OWN * RS;         // [64][RS]
  float *Vs = Ks + BB_TILE * RS;        // [64][RS]
  float *Ps = Vs + BB_TILE * RS;        // [32][68] dS
  float *lse_s = Ps + BB_OWN * BB_PS;   // [32]
  float *del_s = lse_s + BB_OWN;        // [32]

  const int b = blockIdx.z, head = blockIdx.y, q0 = blockIdx.x * BB_OWN;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int d = nheads * hd, nv = hd >> 2;
  const int len = min(max(lengths[b], 0), S);
  // ragged layout (offsets != NULL): episode b owns rows offsets[b] .. offsets[b] + len - 1 and nothing beyond
  const int64_t row0 = offsets ? (int64_t)offsets[b] : (int64_t)b * S;
  const int Sq = offsets ? len : S;  // rows of this episode that exist in memory
  const int cg = NCW == 1 ? tid % nv : tid & 31, rg = NCW == 1 ? tid / nv : tid >> 5;
  const bool out_thread = rg < BB_OWN / 4;
  // column of chunk c; a thread whose cg + 32 c lies past the head computes the last column again and does not store it
  auto col = [&](int c) { return c == 0 ? cg : min(cg + 32 * c, nv - 1); };
  auto col_ok = [&](int c) { return c == 0 || cg + 32 * c < nv; };
  const int64_t stat0 = ((int64_t)b * nheads + head) * S;

  if (q0 >= len) {
    if (out_thread) {
#pragma unroll
      for (int c = 0; c < NCW; ++c) {
        if (!col_ok(c)) continue;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int i = q0 + rg * 4 + r;
          if (i < Sq) reinterpret_cast<float4 *>(dqkv + (row0 + i) * ld + head * hd)[col(c)] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    }
    if (tid < BB_OWN && q0 + tid < S) delta[stat0 + q0 + tid] = 0.0f;
    return;
  }

  const float scale = sqrtf((float)hd);
  for (int idx = tid; idx < BB_OWN * nv; idx += BB_THREADS) {
    const int r = idx / nv, c = idx % nv;
    float4 q = make_float4(0.f, 0.f, 0.f, 0.f), g = q;
    if (q0 + r < len) {
      q = __ldg(reinterpret_cast<const float4 *>(qkv + (row0 + q0 + r) * ld + head * hd) + c);
      q.x /= scale; q.y /= scale; q.z /= scale; q.w /= scale;
      g = __ldg(reinterpret_cast<const float4 *>(dO + (row0 + q0 + r) * d + head * hd) + c);
    }
    reinterpret_cast<float4 *>(Qs + r * RS)[c] = q;
    reinterpret_cast<float4 *>(Gs + r * RS)[c] = g;
  }
  // delta_i = sum_c dO[i,c] O[i,c]   (4 rows per warp)
#pragma unroll
  for (int rr = 0; rr < 4; ++rr) {
    const int r = warp * 4 + rr, i = q0 + r;
    float s = 0.0f;
    if (i < len)
      for (int c = lane; c < hd; c += 32)
        s = fmaf(__ldg(dO + (row0 + i) * d + head * hd + c), __ldg(o + (row0 + i) * d + head * hd + c), s);
    s = warp_sum(s);
    if (lane == 0) {
      del_s[r] = s;
      lse_s[r] = (i < len) ? __ldg(lse + stat0 + i) : 0.0f;
      if (i < S) delta[stat0 + i] = s;
    }
  }

  float acc_o[NCW][4][4];
#pragma unroll
  for (int n = 0; n < NCW; ++n)
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc_o[n][r][c] = 0.0f;

  const int kbeg = max(0, q0 - w), kend = min(len, q0 + BB_OWN + w);
  const int qg = tid >> 4, kg = tid & 15;
  for (int k0 = kbeg; k0 < kend; k0 += BB_TILE) {
    __syncthreads();  // previous tile fully consumed (and, first time, Qs/Gs/stat rows visible)
    for (int idx = tid; idx < BB_TILE * nv; idx += BB_THREADS) {
      const int r = idx / nv, c = idx % nv;
      float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
      if (k0 + r < kend) {
        const float *base = qkv + (row0 + k0 + r) * ld + head * hd;
        kv = __ldg(reinterpret_cast<const float4 *>(base + d) + c);
        vv = __ldg(reinterpret_cast<const float4 *>(base + 2 * d) + c);
      }
      reinterpret_cast<float4 *>(Ks + r * RS)[c] = kv;
      reinterpret_cast<float4 *>(Vs + r * RS)[c] = vv;
    }
    __syncthreads();
    {
      float as[2][4], ap[2][4];
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int j = 0; j < 4; ++j) { as[a][j] = 0.0f; ap[a][j] = 0.0f; }
      for (int c = 0; c < nv; ++c) {
        const float4 x0 = reinterpret_cast<const float4 *>(Qs + qg * RS)[c];
        const float4 x1 = reinterpret_cast<const float4 *>(Qs + (qg + 16) * RS)[c];
        const float4 g0 = reinterpret_cast<const float4 *>(Gs + qg * RS)[c];
        const float4 g1 = reinterpret_cast<const float4 *>(Gs + (qg + 16) * RS)[c];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 kk = reinterpret_cast<const float4 *>(Ks + (kg + 16 * j) * RS)[c];
          const float4 vv = reinterpret_cast<const float4 *>(Vs + (kg + 16 * j) * RS)[c];
          as[0][j] = dot4(x0, kk, as[0][j]);
          as[1][j] = dot4(x1, kk, as[1][j]);
          ap[0][j] = dot4(g0, vv, ap[0][j]);
          ap[1][j] = dot4(g1, vv, ap[1][j]);
        }
      }
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        const int r = qg + 16 * a, i = q0 + r;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int kj = k0 + kg + 16 * j;
          const bool ok = (i < len) && (kj < kend) && (kj >= i - w) && (kj <= i + w);
          const float p = ok ? expf(as[a][j] - lse_s[r]) : 0.0f;
          float dp = ap[a][j];
          if (DROP) dp *= attn_keep_scale(seed, (uint32_t)(b * nheads + head), (uint32_t)i, (uint32_t)kj, p24, inv_keep);
          Ps[r * BB_PS + kg + 16 * j] = p * (dp - del_s[r]);
        }
      }
    }
    __syncthreads();
    if (out_thread) {
#pragma unroll 4
      for (int k4 = 0; k4 < BB_TILE / 4; ++k4) {
        float4 p[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) p[r] = reinterpret_cast<const float4 *>(Ps + (rg * 4 + r) * BB_PS)[k4];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
          for (int n = 0; n < NCW; ++n) {
            const float4 kv = reinterpret_cast<const float4 *>(Ks + (4 * k4 + kk) * RS)[col(n)];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              const float pk = kk == 0 ? p[r].x : kk == 1 ? p[r].y : kk == 2 ? p[r].z : p[r].w;
              acc_o[n][r][0] = fmaf(pk, kv.x, acc_o[n][r][0]);
              acc_o[n][r][1] = fmaf(pk, kv.y, acc_o[n][r][1]);
              acc_o[n][r][2] = fmaf(pk, kv.z, acc_o[n][r][2]);
              acc_o[n][r][3] = fmaf(pk, kv.w, acc_o[n][r][3]);
            }
          }
        }
      }
    }
  }
  if (out_thread) {
#pragma unroll
    for (int n = 0; n < NCW; ++n) {
      if (!col_ok(n)) continue;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int i = q0 + rg * 4 + r;
        if (i >= Sq) continue;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < len)
          v = make_float4(acc_o[n][r][0] / scale, acc_o[n][r][1] / scale, acc_o[n][r][2] / scale, acc_o[n][r][3] / scale);
        reinterpret_cast<float4 *>(dqkv + (row0 + i) * ld + head * hd)[col(n)] = v;
      }
    }
  }
}

template <bool DROP, int NCW>
__global__ void __launch_bounds__(BB_THREADS, NCW == 1 ? 2 : 1)
    band_attn_bwd_dkv_kernel(const float *__restrict__ qkv, int64_t ld, const float *__restrict__ dO,
                             const float *__restrict__ lse, const float *__restrict__ delta,
                             const int32_t *__restrict__ lengths, const int32_t *__restrict__ offsets, int S,
                             int nheads, int hd, int w, float *__restrict__ dqkv, uint32_t p24, float inv_keep,
                             uint64_t seed) {
  extern __shared__ __align__(16) float sm[];
  const int RS = bb_row_stride(hd);
  float *Ks = sm;                        // [32][RS] own keys
  float *Vs = Ks + BB_OWN * RS;          // [32][RS] own values
  float *Qs = Vs + BB_OWN * RS;          // [64][RS] scaled queries of the tile
  float *Gs = Qs + BB_TILE * RS;         // [64][RS] dO of the tile
  float *Pt = Gs + BB_TILE * RS;         // [32][68] P^T
  float *St = Pt + BB_OWN * BB_PS;       // [32][68] dS^T
  float *lse_s = St + BB_OWN * BB_PS;    // [64]
  float *del_s = lse_s + BB_TILE;        // [64]

  const int b = blockIdx.z, head = blockIdx.y, k0 = blockIdx.x * BB_OWN;
  const int tid = threadIdx.x;
  const int d = nheads * hd, nv = hd >> 2;
  const int len = min(max(lengths[b], 0), S);
  // ragged layout (offsets != NULL): episode b owns rows offsets[b] .. offsets[b] + len - 1 and nothing beyond
  const int64_t row0 = offsets ? (int64_t)offsets[b] : (int64_t)b * S;
  const int Sq = offsets ? len : S;  // rows of this episode that exist in memory
  const int cg = NCW == 1 ? tid % nv : tid & 31, rg = NCW == 1 ? tid / nv : tid >> 5;
  const bool out_thread = rg < BB_OWN / 4;
  // column of chunk c; a thread whose cg + 32 c lies past the head computes the last column again and does not store it
  auto col = [&](int c) { return c == 0 ? cg : min(cg + 32 * c, nv - 1); };
  auto col_ok = [&](int c) { return c == 0 || cg + 32 * c < nv; };
  const int64_t stat0 = ((int64_t)b * nheads + head) * S;

  float dk[NCW][4][4], dv[NCW][4][4];
#pragma unroll
  for (int n = 0; n < NCW; ++n)
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) { dk[n][r][c] = 0.0f; dv[n][r][c] = 0.0f; }

  if (k0 < len) {
    for (int idx = tid; idx < BB_OWN * nv; idx += BB_THREADS) {
      const int r = idx / nv, c = idx % nv;
      float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
      if (k0 + r < len) {
        const float *base = qkv + (row0 + k0 + r) * ld + head * hd;
        kv = __ldg(reinterpret_cast<const float4 *>(base + d) + c);
        vv = __ldg(reinterpret_cast<const float4 *>(base + 2 * d) + c);
      }
      reinterpret_cast<float4 *>(Ks + r * RS)[c] = kv;
      reinterpret_cast<float4 *>(Vs + r * RS)[c] = vv;
    }
    const float scale = sqrtf((float)hd);
    const int qbeg = max(0, k0 - w), qend = min(len, k0 + BB_OWN + w);
    const int kgq = tid >> 4, qq = tid & 15;
    for (int t0 = qbeg; t0 < qend; t0 += BB_TILE) {
      __syncthreads();
      for (int idx = tid; idx < BB_TILE * nv; idx += BB_THREADS) {
        const int r = idx / nv, c = idx % nv;
        float4 q = make_float4(0.f, 0.f, 0.f, 0.f), g = q;
        if (t0 + r < qend) {
          q = __ldg(reinterpret_cast<const float4 *>(qkv + (row0 + t0 + r) * ld + head * hd) + c);
          q.x /= scale; q.y /= scale; q.z /= scale; q.w /= scale;
          g = __ldg(reinterpret_cast<const float4 *>(dO + (row0 + t0 + r) * d + head * hd) + c);
        }
        reinterpret_cast<float4 *>(Qs + r * RS)[c] = q;
        reinterpret_cast<float4 *>(Gs + r * RS)[c] = g;
      }
      if (tid < BB_TILE) {
        const bool ok = t0 + tid < qend;
        lse_s[tid] = ok ? __ldg(lse + stat0 + t0 + tid) : 0.0f;
        del_s[tid] = ok ? __ldg(delta + stat0 + t0 + tid) : 0.0f;
      }
      __syncthreads();
      {
        float as[2][4], ap[2][4];
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int j = 0; j < 4; ++j) { as[a][j] = 0.0f; ap[a][j] = 0.0f; }
        for (int c = 0; c < nv; ++c) {
          const float4 x0 = reinterpret_cast<const float4 *>(Ks + kgq * RS)[c];
          const float4 x1 = reinterpret_cast<const float4 *>(Ks + (kgq + 16) * RS)[c];
          const float4 v0 = reinterpret_cast<const float4 *>(Vs + kgq * RS)[c];
          const float4 v1 = reinterpret_cast<const float4 *>(Vs + (kgq + 16) * RS)[c];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 qv = reinterpret_cast<const float4 *>(Qs + (qq + 16 * j) * RS)[c];
            const float4 gv = reinterpret_cast<const float4 *>(Gs + (qq + 16 * j) * RS)[c];
            as[0][j] = dot4(x0, qv, as[0][j]);
            as[1][j] = dot4(x1, qv, as[1][j]);
            ap[0][j] = dot4(v0, gv, ap[0][j]);
            ap[1][j] = dot4(v1, gv, ap[1][j]);
          }
        }
#pragma unroll
        for (int a = 0; a < 2; ++a) {
          const int r = kgq + 16 * a, kj = k0 + r;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int qi = qq + 16 * j, i = t0 + qi;
            const bool ok = (kj < len) && (i < qend) && (kj >= i - w) && (kj <= i + w);
            const float p = ok ? expf(as[a][j] - lse_s[qi]) : 0.0f;
            float m = 1.0f;
            if (DROP) m = attn_keep_scale(seed, (uint32_t)(b * nheads + head), (uint32_t)i, (uint32_t)kj, p24, inv_keep);
            Pt[r * BB_PS + qi] = p * m;
            St[r * BB_PS + qi] = p * (m * ap[a][j] - del_s[qi]);
          }
        }
      }
      __syncthreads();
      if (out_thread) {
#pragma unroll 2
        for (int q4 = 0; q4 < BB_TILE / 4; ++q4) {
          float4 p[4], s[4];
#pragma unroll
          for (int r = 0; r < 4; ++r) {
            p[r] = reinterpret_cast<const float4 *>(Pt + (rg * 4 + r) * BB_PS)[q4];
            s[r] = reinterpret_cast<const float4 *>(St + (rg * 4 + r) * BB_PS)[q4];
          }
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
            for (int n = 0; n < NCW; ++n) {
              const float4 gv = reinterpret_cast<const float4 *>(Gs + (4 * q4 + kk) * RS)[col(n)];
              const float4 qv = reinterpret_cast<const float4 *>(Qs + (4 * q4 + kk) * RS)[col(n)];
#pragma unroll
              for (int r = 0; r < 4; ++r) {
                const float pk = kk == 0 ? p[r].x : kk == 1 ? p[r].y : kk == 2 ? p[r].z : p[r].w;
                const float sk = kk == 0 ? s[r].x : kk == 1 ? s[r].y : kk == 2 ? s[r].z : s[r].w;
                dv[n][r][0] = fmaf(pk, gv.x, dv[n][r][0]); dv[n][r][1] = fmaf(pk, gv.y, dv[n][r][1]);
                dv[n][r][2] = fmaf(pk, gv.z, dv[n][r][2]); dv[n][r][3] = fmaf(pk, gv.w, dv[n][r][3]);
                dk[n][r][0] = fmaf(sk, qv.x, dk[n][r][0]); dk[n][r][1] = fmaf(sk, qv.y, dk[n][r][1]);
                dk[n][r][2] = fmaf(sk, qv.z, dk[n][r][2]); dk[n][r][3] = fmaf(sk, qv.w, dk[n][r][3]);
              }
            }
          }
        }
      }
    }
  }
  if (out_thread) {
#pragma unroll
    for (int n = 0; n < NCW; ++n) {
      if (!col_ok(n)) continue;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int kj = k0 + rg * 4 + r;
        if (kj >= Sq) continue;
        float *base = dqkv + (row0 + kj) * ld + head * hd;
        reinterpret_cast<float4 *>(base + d)[col(n)] = make_float4(dk[n][r][0], dk[n][r][1], dk[n][r][2], dk[n][r][3]);
        reinterpret_cast<float4 *>(base + 2 * d)[col(n)] = make_float4(dv[n][r][0], dv[n][r][1], dv[n][r][2], dv[n][r][3]);
      }
    }
  }
}

static unsigned ew_grid2(int64_t total) {
  int64_t g = (total + 255) / 256;
  const int64_t cap = (int64_t)kNumSMs * 16;
  return (unsigned)(g < cap ? (g > 0 ? g : 1) : cap);
}

static int ln_chunks(int M) {
  const int want = kNumSMs * 4;
  return M < want ? M : want;
}

}  // namespace mts

using namespace mts;

extern "C" int64_t mts_ln_bwd_ws_bytes(int M, int d) {
  if (M <= 0 || d <= 0) return 0;
  return (int64_t)ln_chunks(M) * 2 * d * (int64_t)sizeof(float);
}

extern "C" int mts_ln_bwd(const float *dy, const float *pre, const float *stats, const float *gamma, int M, int d,
                          float *dx, float *dx_hi, float *dx_lo, int Kp, float *dgamma, float *dbeta, void *ws,
                          void *stream) {
  MTS_REQUIRE(dy && pre && stats && gamma && dx && dgamma && dbeta && ws, MTS_E_BADARG, "ln_bwd: null pointer");
  MTS_REQUIRE(M > 0 && d > 0, MTS_E_BADARG, "ln_bwd: empty shape");
  MTS_REQUIRE(d % 4 == 0 && d <= 128 * LNB_MAXV, MTS_E_UNSUPPORTED, "ln_bwd: width must be a multiple of 4 and <= 2048");
  MTS_REQUIRE(!(dx_hi && !dx_lo), MTS_E_BADARG, "ln_bwd: hi without lo");
  MTS_REQUIRE(!(dx_lo && !dx_hi) || Kp == d, MTS_E_BADARG, "ln_bwd: dx can only stand in for hi when Kp == d");
  MTS_REQUIRE(!dx_lo || (Kp % 32 == 0 && Kp >= d), MTS_E_BADARG, "ln_bwd: Kp");
  cudaStream_t st = (cudaStream_t)stream;
  const int chunks = ln_chunks(M);
  const int rows_per = (M + chunks - 1) / chunks;
  const int used = (M + rows_per - 1) / rows_per;
  ln_bwd_param_kernel<<<used, 256, 0, st>>>(dy, pre, stats, M, d, rows_per, (float *)ws);
  ln_bwd_param_final_kernel<<<(2 * d + 255) / 256, 256, 0, st>>>((const float *)ws, used, d, dgamma, dbeta);
  const unsigned grid = (unsigned)min((int64_t)(M + 7) / 8, (int64_t)kNumSMs * 8);
  ln_bwd_dx_kernel<<<grid, 256, 0, st>>>(dy, pre, stats, gamma, M, d, dx, dx_hi, dx_lo, Kp);
  MTS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mts_gelu_bwd(const float *dz, const float *zp, int rows, int cols, int Kp, float *dzp, float *hi,
                            float *lo, void *stream) {
  MTS_REQUIRE(dz && zp && dzp && hi && lo, MTS_E_BADARG, "gelu_bwd: null pointer");
  MTS_REQUIRE(rows > 0 && cols > 0 && Kp % 32 == 0 && Kp >= cols, MTS_E_BADARG, "gelu_bwd: bad shape");
  gelu_bwd_kernel<<<ew_grid2((int64_t)rows * Kp), 256, 0, (cudaStream_t)stream>>>(dz, zp, rows, cols, Kp, dzp, hi, lo);
  MTS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mts_embed_bwd(const float *dpre, int B, int S, int d, float *dpos, const int32_t *lengths,
                             const int32_t *offsets, void *stream) {
  MTS_REQUIRE(dpre && dpos, MTS_E_BADARG, "embed_bwd: null pointer");
  MTS_REQUIRE(!offsets || lengths, MTS_E_BADARG, "embed_bwd: ragged rows need the lengths");
  MTS_REQUIRE(B > 0 && S > 0 && d > 0 && d % 4 == 0, MTS_E_BADARG, "embed_bwd: bad shape");
  embed_bwd_kernel<<<ew_grid2((int64_t)S * (d / 4)), 256, 0, (cudaStream_t)stream>>>(dpre, B, S, d, dpos, lengths, offsets);
  MTS_LAUNCH_CHECK();
  return 0;
}

template <bool DROP, int NCW>
static int band_attn_bwd_launch(const float *qkv, int64_t ld, const float *o, const float *d_o, const float *lse,
                                const int32_t *lengths, const int32_t *offsets, int B, int S, int nheads, int hd, int w,
                                float *dqkv, float *delta_ws, float p_drop, uint64_t seed, void *stream) {
  const int RS = bb_row_stride(hd);
  const size_t smem_dq = sizeof(float) * ((size_t)(2 * BB_OWN + 2 * BB_TILE) * RS + BB_OWN * BB_PS + 2 * BB_OWN);
  const size_t smem_dkv = sizeof(float) * ((size_t)(2 * BB_OWN + 2 * BB_TILE) * RS + 2 * BB_OWN * BB_PS + 2 * BB_TILE);
  MTS_PER_DEVICE(size_t, set_dq);   // one pair per instantiation and device
  MTS_PER_DEVICE(size_t, set_dkv);
  if (smem_dq > set_dq) {
    MTS_CUDA(cudaFuncSetAttribute(band_attn_bwd_dq_kernel<DROP, NCW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_dq));
    set_dq = smem_dq;
  }
  if (smem_dkv > set_dkv) {
    MTS_CUDA(cudaFuncSetAttribute(band_attn_bwd_dkv_kernel<DROP, NCW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_dkv));
    set_dkv = smem_dkv;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid((S + BB_OWN - 1) / BB_OWN, nheads, B);
  const uint32_t p24 = DROP ? attn_drop_p24(p_drop) : 0u;
  const float inv_keep = DROP ? 1.0f / (1.0f - p_drop) : 1.0f;
  band_attn_bwd_dq_kernel<DROP, NCW><<<grid, BB_THREADS, smem_dq, st>>>(qkv, ld, o, d_o, lse, lengths, offsets, S, nheads, hd, w,
                                                                   dqkv, delta_ws, p24, inv_keep, seed);
  band_attn_bwd_dkv_kernel<DROP, NCW><<<grid, BB_THREADS, smem_dkv, st>>>(qkv, ld, d_o, lse, delta_ws, lengths, offsets, S, nheads,
                                                                     hd, w, dqkv, p24, inv_keep, seed);
  MTS_LAUNCH_CHECK();
  return 0;
}

extern "C" int mts_band_attn_bwd_dropout(const float *qkv, int64_t ld, const float *o, const float *d_o, const float *lse,
                                         const int32_t *lengths, const int32_t *offsets, int B, int S, int nheads, int hd,
                                         int w, float *dqkv, float *delta_ws, float p_drop, uint64_t seed, void *stream) {
  MTS_REQUIRE(qkv && o && d_o && lse && lengths && dqkv && delta_ws, MTS_E_BADARG, "band_attn_bwd: null pointer");
  MTS_REQUIRE(B > 0 && S > 0 && nheads > 0 && hd > 0 && w >= 0, MTS_E_BADARG, "band_attn_bwd: bad shape");
  MTS_REQUIRE(hd % 4 == 0 && hd <= 256, MTS_E_UNSUPPORTED, "band_attn_bwd: head dim must be a multiple of 4 and <= 256");
  MTS_REQUIRE(ld % 4 == 0 && ld >= 3 * nheads * hd, MTS_E_BADARG, "band_attn_bwd: qkv row stride");
  MTS_REQUIRE(p_drop >= 0.0f && p_drop < 1.0f, MTS_E_BADARG, "band_attn_bwd: dropout probability must be in [0, 1)");
  MTS_REQUIRE(p_drop == 0.0f || S <= (1 << 20), MTS_E_UNSUPPORTED, "band_attn_bwd: dropout indices need S <= 2^20");
  if (hd > 128) {
    if (p_drop > 0.0f)
      return band_attn_bwd_launch<true, 2>(qkv, ld, o, d_o, lse, lengths, offsets, B, S, nheads, hd, w, dqkv, delta_ws, p_drop, seed, stream);
    return band_attn_bwd_launch<false, 2>(qkv, ld, o, d_o, lse, lengths, offsets, B, S, nheads, hd, w, dqkv, delta_ws, 0.0f, 0ull, stream);
  }
  if (p_drop > 0.0f)
    return band_attn_bwd_launch<true, 1>(qkv, ld, o, d_o, lse, lengths, offsets, B, S, nheads, hd, w, dqkv, delta_ws, p_drop, seed, stream);
  return band_attn_bwd_launch<false, 1>(qkv, ld, o, d_o, lse, lengths, offsets, B, S, nheads, hd, w, dqkv, delta_ws, 0.0f, 0ull, stream);
}

extern "C" int mts_band_attn_bwd(const float *qkv, int64_t ld, const float *o, const float *d_o, const float *lse,
                                 const int32_t *lengths, const int32_t *offsets, int B, int S, int nheads, int hd, int w,
                                 float *dqkv, float *delta_ws, void *stream) {
  return mts_band_attn_bwd_dropout(qkv, ld, o, d_o, lse, lengths, offsets, B, S, nheads, hd, w, dqkv, delta_ws, 0.0f, 0ull, stream);
}
