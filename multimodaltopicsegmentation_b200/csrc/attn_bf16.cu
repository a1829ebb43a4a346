// Banded (windowed) self-attention, forward, over bf16 q/k/v (inference under the bf16 precision switch).
// Same contract as mts_band_attn_fwd (HF LongformerSelfAttention, modeling_longformer.py:481-639; call site
// models/RestrictedTransformerLayer.py:131): softmax over |i - j| <= w, j < len_b of (q_i / sqrt(hd)) . k_j, exact zeros for
// padded queries (:578) -- here with q, k, v given as bf16 and both products on kind::f16 (bf16) MMAs, fp32 accumulation:
//     S = Q K^T   (A = Q tile in shared memory, B = K tile; fp32 in tensor memory)
//     O += P V    (A = bf16(P) in tensor memory, .ts form; B = V tile, MN-major)
// The softmax itself (masks, scale 1 / sqrt(hd), lazy rescale, row sums, log-sum-exp) is fp32, as in attn_tc.cu.
//
// Operands arrive by TMA straight in the layouts the MMAs read -- no CUDA-core pass touches Q, K or V:
//   Q tile: 128 rows x 64 bf16 per box, K-major SWIZZLE_128B (one plane per 64 head columns)
//   K tile: 64 keys x 64 bf16 per box, K-major SWIZZLE_128B (N = keys, K = head dim)
//   V tile: the same boxes, read as MN-major SWIZZLE_128B (N = head dim, K = keys): one 128-byte swizzle row per key
// K and V are double-buffered (the fp32 kernel's raw + correction planes took that room).  Q is read by the MMA from shared
// memory (.ss form): the .ts form would need the worker warps to stage Q through registers into tensor memory (~5.5 k cycles per
// item in attn_tc.cu), while the TMA lands the tile in shared memory with no worker involvement; S costs HD / 16 MMAs per key tile.
//
// Tensor memory (512 columns): S tiles [128,192) [192,256) fp32 | P tiles [256,288) [288,320) bf16 pairs | O [384, 384+HD);
// heads wider than 128 move S to [0,128) and P to [128,192) so that O [256, 256+HD) fits (512 columns at HD 256).
// Warps: 8 uniform worker warps (softmax + epilogue, as in attn_tc.cu), warp 8 MMA issuer, warps 9 / 10 / 11 TMA loaders of
// K / V / Q.  Per key tile a worker warp only reads S, masks, exchanges row maxima with its partner warp and writes P.
#include <stdlib.h>

#include "attn_band.cuh"

namespace mts {
namespace atc {

template <int HD>
struct Cfg16 {
  static_assert(HD % 16 == 0 && HD >= 16 && HD <= 256, "head dim: multiple of 16, at most 256");
  static constexpr uint32_t COL_S = HD <= 128 ? 128 : 0, COL_P = HD <= 128 ? 256 : 128, COL_O = HD <= 128 ? 384 : 256;
  static constexpr int NP = (HD + 63) / 64;    // 64-column (128-byte) planes of a bf16 operand
  static constexpr int NC = HD / 16;           // 16-column chunks per row
  static constexpr int Q_BYTES = NP * BQ * 128;
  static constexpr int T_BYTES = NP * KT * 128;   // one K or V tile
  static constexpr int OFF_Q = 0;
  static constexpr int OFF_K = OFF_Q + Q_BYTES;         // [2] K buffers
  static constexpr int OFF_V = OFF_K + 2 * T_BYTES;     // [2] V buffers
  static constexpr int OFF_TR = OFF_V + 2 * T_BYTES;
  static constexpr int TR_BYTES = 8 * 32 * TRS * 4;
  static constexpr int OFF_MX = OFF_TR + TR_BYTES;           // [2 tile parity][2 column halves][128] partial row maxima
  static constexpr int OFF_LS = OFF_MX + 2 * 2 * BQ * 4;     // [2 column halves][128] partial row sums
  static constexpr int OFF_BAR = OFF_LS + 2 * BQ * 4;
  static constexpr int OFF_META = OFF_BAR + 16 * 8 + 16;
  static constexpr int USED = OFF_META + 2 * META_B * 4;
  // every CTA allocates all 512 TMEM columns, so two CTAs must never share an SM: ask for more than half its shared memory
  static constexpr int SMEM = (USED + 1024) > 120 * 1024 ? (USED + 1024) : 120 * 1024;
  static_assert(SMEM <= 227 * 1024, "shared memory of one CTA");
};

enum { C_QFULL = 0, C_QFREE, C_KFULL0, C_KFULL1, C_KEMPTY0, C_KEMPTY1, C_VFULL0, C_VFULL1, C_VEMPTY0, C_VEMPTY1,
       C_SFULL0, C_SFULL1, C_PREADY0, C_PREADY1, C_ODONE, C_OFREE, C_COUNT };
static_assert(C_COUNT <= 16, "barrier block holds 16 mbarriers");

template <int HD>
__global__ void __launch_bounds__(THREADS, 1)
    band_attn_fwd_bf16_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_kv,
                              const int32_t *__restrict__ lengths, const int32_t *__restrict__ offsets, int B, int S, int nheads,
                              int w, float *__restrict__ out, float *__restrict__ out_lo, float *__restrict__ lse) {
  using C = Cfg16<HD>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = tc::s_u32(smem);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + C::OFF_BAR);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 16);
  int32_t *meta_p = reinterpret_cast<int32_t *>(smem + C::OFF_META);
  const uint32_t mx_s = sbase + C::OFF_MX, ls_s = sbase + C::OFF_LS;

  const int lane = threadIdx.x & 31;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int d = nheads * HD;
  Seq sq;
  sq.nheads = nheads;
  sq.n_qb = (S + BQ - 1) / BQ;
  sq.S = S;
  sq.w = w;
  sq.n_items = B * sq.n_qb * nheads;
  sq.step = gridDim.x;
  sq.s_head = sq.step % nheads;
  sq.s_qb = (sq.step / nheads) % sq.n_qb;
  sq.s_b = (sq.step / nheads) / sq.n_qb;
  sq.lengths = lengths;
  sq.offsets = offsets;
  sq.meta = sbase + C::OFF_META;
#define BAR(i) (sbase + (uint32_t)(C::OFF_BAR + 8 * (i)))

  if (threadIdx.x == 0) {
    tc::bar_init(BAR(C_QFULL), 1);
    tc::bar_init(BAR(C_QFREE), 1);
    for (int b = 0; b < 2; ++b) {
      tc::bar_init(BAR(C_KFULL0 + b), 1);
      tc::bar_init(BAR(C_KEMPTY0 + b), 1);
      tc::bar_init(BAR(C_VFULL0 + b), 1);
      tc::bar_init(BAR(C_VEMPTY0 + b), 1);
      tc::bar_init(BAR(C_SFULL0 + b), 1);
      tc::bar_init(BAR(C_PREADY0 + b), WORKERS);
    }
    tc::bar_init(BAR(C_ODONE), 1);
    tc::bar_init(BAR(C_OFREE), WORKERS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) tc::tmem_alloc<512>(tc::s_u32(tmem_slot));
  for (int e = threadIdx.x; e < min(B, META_B); e += THREADS) {
    meta_p[e] = lengths[e];
    meta_p[META_B + e] = offsets ? offsets[e] : 0;
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 8) {
    // ======================================= worker warps =======================================
    const int q = warp & 3, ch = warp >> 2;          // TMEM lane quarter, column half
    const int r = q * 32 + lane;                     // my query row inside the item
    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
    const uint32_t tr = sbase + (uint32_t)(C::OFF_TR + warp * 32 * TRS * 4);
    const float inv_scale = 1.0f / sqrtf((float)HD);   // HF divides q by sqrt(head_dim) (:513); applied to the fp32 scores here
    uint32_t item_g = 0, tile_g = 0;                 // items / tiles completed
    Item it;
    for (item_first(it, sq, blockIdx.x); it.idx < sq.n_items; item_step(it, sq)) {
      float inv = 0.0f, lse_v = 0.0f;
      if (it.active) {
        const int i = it.q0 + r;
        float m_run = -INFINITY, l_run = 0.0f;
#pragma unroll 1
        for (int t = 0; t < it.nt; ++t) {
          const int buf = tile_g & 1;
          const int k0 = tile_k0(it, t) + 32 * ch;     // first key of my column half
          // valid column range [clo, clo + nvalid) of my row inside my half: band |i - j| <= w, j < kend (<= len), and not a
          // key the previous tile has covered already (the last tile's box is shifted up to end at kend)
          const int clo = max(max(0, i - w - k0), it.kbeg + t * KT - k0);
          const int chi = (i < it.len) ? min(it.kend - k0, i + w + 1 - k0) : 0;
          const unsigned nvalid = (unsigned)max(min(chi, 32) - clo, 0);
          bar_wait(BAR(C_SFULL0 + buf), (tile_g >> 1) & 1);
          tc::tc_fence_after();
          float s[32];
          tmem_ld32_nowait(trow + C::COL_S + 64 * buf + 32 * ch, s);
          tmem_wait_ld();
          // 16-key blocks that no row of this warp can see are not evaluated: their probabilities are stored as zeros
          unsigned live = 0;
#pragma unroll
          for (int blk = 0; blk < 2; ++blk)
            if (__any_sync(0xffffffffu, clo < 16 * blk + 16 && chi > 16 * blk)) live |= 1u << blk;
          float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
          for (int blk = 0; blk < 2; ++blk) {
            if (!(live & (1u << blk))) continue;
#pragma unroll
            for (int e = 0; e < 16; ++e) {
              const int c = 16 * blk + e;
              s[c] = ((unsigned)(c - clo) < nvalid) ? s[c] * inv_scale : -INFINITY;
              mx4[e & 3] = fmaxf(mx4[e & 3], s[c]);
            }
          }
          float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
          sts_f32(mx_s + 4 * ((buf * 2 + ch) * BQ + r), mx);
          pair_sync(q);
          mx = fmaxf(mx, lds_f32(mx_s + 4 * ((buf * 2 + (ch ^ 1)) * BQ + r)));
          float alpha = 1.0f;
          if (mx > m_run + RESCALE_TH) {
            if (m_run != -INFINITY) { alpha = ex2f((m_run - mx) * LOG2E); l_run *= alpha; }
            m_run = mx;
          }
          if (t > 0 && __any_sync(0xffffffffu, alpha != 1.0f)) {
            // rare: rescale my column half of O; the previous P V (tile tile_g - 1, V buffer (tile_g - 1) & 1) must be complete.
            // The S product of this tile was issued after the P V of tile tile_g - 2, so that barrier is at most one phase behind.
            const uint32_t pv = tile_g - 1;
            bar_wait(BAR(C_VEMPTY0 + (pv & 1)), (pv >> 1) & 1);
            tc::tc_fence_after();
#pragma unroll 1
            for (int c = ch; c < C::NC; c += 2) {
              float v[16];
              uint32_t u[16];
              tmem_ld16_nowait(trow + C::COL_O + 16 * c, v);
              tmem_wait_ld();
#pragma unroll
              for (int e = 0; e < 16; ++e) u[e] = __float_as_uint(v[e] * alpha);
              tmem_st16(trow + C::COL_O + 16 * c, u);
            }
          }
          const float mb = (m_run == -INFINITY) ? 0.0f : -m_run * LOG2E;
          float ps4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
          uint32_t pb[16];   // bf16(p) of my 32 keys, two per 32-bit column (the A operand of P V, K = 16 per 8 columns)
#pragma unroll
          for (int blk = 0; blk < 2; ++blk) {
            if (live & (1u << blk)) {
#pragma unroll
              for (int e = 0; e < 16; e += 2) {
                const float p0 = ex2f(fmaf(s[16 * blk + e], LOG2E, mb)), p1 = ex2f(fmaf(s[16 * blk + e + 1], LOG2E, mb));
                ps4[(e >> 1) & 3] += p0 + p1;
                pb[8 * blk + (e >> 1)] = bf16x2_bits(p0, p1);
              }
            } else {
#pragma unroll
              for (int e = 0; e < 8; ++e) pb[8 * blk + e] = 0u;
            }
          }
          // P buffer `buf` was last read by the P V of tile tile_g - 2, complete before this tile's S (see C_SFULL above)
          tmem_st16(trow + C::COL_P + 32 * buf + 16 * ch, pb);
          l_run += (ps4[0] + ps4[1]) + (ps4[2] + ps4[3]);
          tc::tmem_wait_st();
          tc::tc_fence_before();
          tc::bar_arrive(BAR(C_PREADY0 + buf));
          ++tile_g;
        }
        sts_f32(ls_s + 4 * (ch * BQ + r), l_run);
        pair_sync(q);
        const float l_tot = l_run + lds_f32(ls_s + 4 * ((ch ^ 1) * BQ + r));
        const bool alive = (i < it.len) && (l_tot > 0.0f);
        inv = alive ? 1.0f / l_tot : 0.0f;
        lse_v = alive ? m_run + logf(l_tot) : 0.0f;
        pair_sync(q);   // ls_s may be rewritten by the next item only after both have read
        bar_wait(BAR(C_ODONE), item_g & 1);   // the last P V of the item has completed
        tc::tc_fence_after();
      }
      // ---- o / l, transposed through the warp's buffer, row-contiguous stores of o and / or its packed operand ----
      // (inactive item = a block of padded queries: exact zeros, HF :578; nothing exists there in the ragged layout)
      if (it.q0 < it.Sq) {
#pragma unroll 1
        for (int c = ch; c < C::NC; c += 2) {
          float v[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) v[e] = 0.0f;
          if (it.active) {
            tmem_ld16_nowait(trow + C::COL_O + 16 * c, v);
            tmem_wait_ld();
          }
#pragma unroll
          for (int j = 0; j < 4; ++j)
            sts128f(tr + 4 * (lane * TRS + 4 * j), make_float4(v[4 * j] * inv, v[4 * j + 1] * inv, v[4 * j + 2] * inv, v[4 * j + 3] * inv));
          __syncwarp();
          // a warp instruction = 8 rows x 64 contiguous bytes (4 lanes per row): o, then the packed operand of the 16-column
          // block (side 0): [bf16(x) 0-7 | bf16(x) 8-15 | bf16(rest) 0-7 | bf16(rest) 8-15], 16 bytes per lane
#pragma unroll
          for (int i2 = 0; i2 < 4; ++i2) {
            const int rr = (lane >> 2) + 8 * i2, pc4 = lane & 3, gi = it.q0 + q * 32 + rr;
            if (gi < it.Sq) {
              const int col = it.head * HD + 16 * c;
              if (out) *reinterpret_cast<float4 *>(out + (it.row0 + gi) * d + col + 4 * pc4) = lds128f(tr + 4 * (rr * TRS + 4 * pc4));
              if (out_lo) {
                float4 e0 = lds128f(tr + 4 * (rr * TRS + 8 * (pc4 & 1)));
                float4 e1 = lds128f(tr + 4 * (rr * TRS + 8 * (pc4 & 1) + 4));
                if (pc4 >= 2) { e0 = rest4(e0); e1 = rest4(e1); }
                *reinterpret_cast<uint4 *>(out_lo + (it.row0 + gi) * d + col + 4 * pc4) = bf16x8(e0, e1);
              }
            }
          }
          __syncwarp();
        }
      }
      if (it.active) {
        tc::tc_fence_before();
        tc::bar_arrive(BAR(C_OFREE));   // my reads of O are done: the next item's first P V may overwrite it
        ++item_g;
      }
      if (ch == 0 && lse && it.q0 + r < S) lse[((int64_t)it.b * nheads + it.head) * S + it.q0 + r] = lse_v;
    }
  } else if (warp == 9 || warp == 10) {
    // ========================= loader warps: K (warp 9) / V (warp 10) tiles by TMA, two buffers each =========================
    if (lane == 0) {
      const bool is_v = warp == 10;
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_kv)) : "memory");
      const uint32_t dst = sbase + (uint32_t)(is_v ? C::OFF_V : C::OFF_K);
      const int full0 = is_v ? C_VFULL0 : C_KFULL0, empty0 = is_v ? C_VEMPTY0 : C_KEMPTY0;
      Cursor cl;
      uint32_t n = 0;
      for (cursor_first(cl, sq, blockIdx.x); cl.valid; cursor_advance(cl, sq), ++n) {
        const uint32_t b = n & 1;
        bar_wait(BAR(empty0 + b), ((n >> 1) & 1) ^ 1);
        tc::bar_expect_tx(BAR(full0 + b), C::T_BYTES);
        const int c0 = (is_v ? 2 : 1) * d + cl.it.head * HD, c1 = (int)cl.it.row0 + tile_k0(cl.it, cl.t);
#pragma unroll
        for (int j = 0; j < C::NP; ++j) tma_load_2d(dst + b * C::T_BYTES + j * (KT * 128), &map_kv, c0 + 64 * j, c1, BAR(full0 + b));
      }
    }
  } else if (warp == 11) {
    // ========================= loader warp: the Q block of every active item by TMA =========================
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_q)) : "memory");
      uint32_t n = 0;
      Item it;
      for (item_first(it, sq, blockIdx.x); it.idx < sq.n_items; item_step(it, sq)) {
        if (!it.active) continue;
        bar_wait(BAR(C_QFREE), (n & 1) ^ 1);   // every S = Q K^T of the previous item has completed
        tc::bar_expect_tx(BAR(C_QFULL), C::Q_BYTES);
#pragma unroll
        for (int j = 0; j < C::NP; ++j)
          tma_load_2d(sbase + C::OFF_Q + j * (BQ * 128), &map_q, it.head * HD + 64 * j, (int)it.row0 + it.q0, BAR(C_QFULL));
        ++n;
      }
    }
  } else if (warp == 8) {
    // =============================== MMA issuer: warp-uniform control flow, one elected lane ===============================
    constexpr uint32_t id_s = tc::idesc_bf16(BQ, KT), id_o = tc::idesc_bf16(BQ, HD) | B_MN_MAJOR;
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
    const bool leader = tc::elect_one();
    const uint64_t q_desc = tc::desc_sw128(sbase + C::OFF_Q), k_desc = tc::desc_sw128(sbase + C::OFF_K);
    const uint64_t v_desc = desc_sw128_mn(sbase + C::OFF_V, KT * 128);
    uint32_t item_g = 0, tile_g = 0, s_cnt = 0, q_seen = 0;
    Cursor cs, cp;   // cs: the next S tile to issue (kept one ahead of the P V position cp)
    cursor_first(cs, sq, blockIdx.x);
    cp = cs;
    bool started = false;
    while (cp.valid) {
      const int nt = cp.it.nt;
#pragma unroll 1
      for (int t = started ? 0 : -1; t < nt; ++t) {
        if (cs.valid) {
          if (cs.t == 0) {   // the tile opens a new item: its Q block must have landed
            bar_wait(BAR(C_QFULL), q_seen & 1);
            ++q_seen;
          }
          const uint32_t kb = s_cnt & 1;
          bar_wait(BAR(C_KFULL0 + kb), (s_cnt >> 1) & 1);
          tc::tc_fence_after();
          const uint32_t d_s = tb + C::COL_S + 64 * (s_cnt & 1);
#pragma unroll
          for (int ks = 0; ks < HD / 16; ++ks) {   // K = 16 bf16 = 32 bytes per MMA inside a 128-byte swizzle row
            const uint64_t ad = desc_add(q_desc, (uint32_t)((ks >> 2) * (BQ * 128) + (ks & 3) * 32));
            const uint64_t bd = desc_add(k_desc, (uint32_t)(kb * C::T_BYTES + (ks >> 2) * (KT * 128) + (ks & 3) * 32));
            if (leader) tc::umma_bf16_ss(d_s, ad, bd, id_s, ks != 0);
          }
          if (leader) {
            tc::umma_commit(BAR(C_SFULL0 + (s_cnt & 1)));
            tc::umma_commit(BAR(C_KEMPTY0 + kb));
            if (cs.t == cs.it.nt - 1) tc::umma_commit(BAR(C_QFREE));   // the item's last S product
          }
          __syncwarp();
          ++s_cnt;
          cursor_advance(cs, sq);
        }
        if (t < 0) {
          started = true;
          continue;
        }
        const uint32_t buf = tile_g & 1;
        bar_wait(BAR(C_PREADY0 + buf), (tile_g >> 1) & 1);
        bar_wait(BAR(C_VFULL0 + buf), (tile_g >> 1) & 1);
        if (t == 0) bar_wait(BAR(C_OFREE), (item_g & 1) ^ 1);   // the previous item's epilogue has read O
        tc::tc_fence_after();
        const uint32_t d_o = tb + C::COL_O;
#pragma unroll
        for (int kg = 0; kg < KT / 16; ++kg) {   // 16 keys = 16 rows of 128 bytes of the V tile per MMA
          const uint64_t bd = desc_add(v_desc, (uint32_t)(buf * C::T_BYTES + kg * 2048));
          if (leader) tc::umma_bf16_ts(d_o, tb + C::COL_P + 32 * buf + 8 * kg, bd, id_o, (t | kg) != 0);
        }
        if (leader) {
          tc::umma_commit(BAR(C_VEMPTY0 + buf));
          if (t == nt - 1) tc::umma_commit(BAR(C_ODONE));
        }
        __syncwarp();
        ++tile_g;
      }
      ++item_g;
      cp.t = nt - 1;
      cursor_advance(cp, sq);
    }
  }
#undef BAR
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc::tc_fence_after();
    tc::tmem_dealloc<512>(tmem_base);
  }
}

// qkv as a 2-D bf16 tensor [rows, 3 d] (row stride ld), boxes of `box_rows` rows x 64 columns (128 bytes, SWIZZLE_128B).  `rows`
// is the true row count of the buffer: a Q box reaching past it (the last query block of the last episode) is zero-filled.
static int make_map_bf16(CUtensorMap *map, const void *qkv, int64_t ld, int width, int64_t rows, int box_rows) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { set_error("band_attn_fwd_bf16: cuTensorMapEncodeTiled not available"); return MTS_E_NODEVICE; }
  cuuint64_t dims[2] = {(cuuint64_t)width, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(qkv), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("band_attn_fwd_bf16: cuTensorMapEncodeTiled failed"); return MTS_E_BADARG; }
  return 0;
}

template <int HD>
static int launch_bf16(const void *qkv, int64_t ld, int64_t rows, const int32_t *lengths, const int32_t *offsets, int B, int S,
                       int nheads, int w, float *out, float *out_lo, float *lse, cudaStream_t st) {
  using C = Cfg16<HD>;
  CUtensorMap map_q, map_kv;
  int rc;
  if ((rc = make_map_bf16(&map_q, qkv, ld, 3 * nheads * HD, rows, BQ))) return rc;
  if ((rc = make_map_bf16(&map_kv, qkv, ld, 3 * nheads * HD, rows, KT))) return rc;
  MTS_CUDA(cudaFuncSetAttribute(band_attn_fwd_bf16_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
  const int n_items = B * ((S + BQ - 1) / BQ) * nheads;
  const int grid = n_items < kNumSMs ? n_items : kNumSMs;
  band_attn_fwd_bf16_kernel<HD><<<grid, THREADS, C::SMEM, st>>>(map_q, map_kv, lengths, offsets, B, S, nheads, w, out, out_lo, lse);
  MTS_LAUNCH_CHECK();
  return 0;
}

}  // namespace atc
}  // namespace mts

using namespace mts;

extern "C" int mts_band_attn_bf16_supported(int hd) {
  return hd == 16 || hd == 32 || hd == 64 || hd == 112 || hd == 128 || (hd >= 144 && hd <= 256 && hd % 16 == 0);
}

extern "C" int mts_band_attn_fwd_bf16(const void *qkv, int64_t ld, int64_t rows, const int32_t *lengths, const int32_t *offsets,
                                      int B, int S, int nheads, int hd, int w, float *out, float *out_lo, int Kp, float *lse,
                                      void *stream) {
  MTS_REQUIRE(qkv && lengths && (out || out_lo), MTS_E_BADARG, "band_attn_fwd_bf16: null pointer");
  MTS_REQUIRE(B > 0 && S > 0 && S <= 4094 && nheads > 0 && hd > 0 && w >= 0, MTS_E_BADARG, "band_attn_fwd_bf16: bad shape");
  MTS_REQUIRE(rows > 0 && rows <= 0x7FFFFFFF && (offsets || rows >= (int64_t)B * S), MTS_E_BADARG, "band_attn_fwd_bf16: row count");
  MTS_REQUIRE(ld % 8 == 0 && ld >= 3 * nheads * hd, MTS_E_BADARG, "band_attn_fwd_bf16: qkv row stride must be a multiple of 8 and >= 3 d");
  MTS_REQUIRE(((uintptr_t)qkv & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)out_lo & 15) == 0, MTS_E_BADARG,
              "band_attn_fwd_bf16: buffers must be 16-byte aligned");
  MTS_REQUIRE(!out_lo || Kp == nheads * hd, MTS_E_UNSUPPORTED, "band_attn_fwd_bf16: the packed output needs Kp == model width");
  MTS_REQUIRE(mts_band_attn_bf16_supported(hd), MTS_E_UNSUPPORTED,
              "band_attn_fwd_bf16: head dim must be one of 16, 32, 64, 112, 128 or 144 .. 256 in steps of 16");
  cudaStream_t st = (cudaStream_t)stream;
  switch (hd) {
#define MTS_BF16_HD(H) \
  case H: return atc::launch_bf16<H>(qkv, ld, rows, lengths, offsets, B, S, nheads, w, out, out_lo, lse, st);
    MTS_BF16_HD(16) MTS_BF16_HD(32) MTS_BF16_HD(64) MTS_BF16_HD(112) MTS_BF16_HD(128)
    MTS_BF16_HD(144) MTS_BF16_HD(160) MTS_BF16_HD(176) MTS_BF16_HD(192) MTS_BF16_HD(208) MTS_BF16_HD(224) MTS_BF16_HD(240)
    MTS_BF16_HD(256)
#undef MTS_BF16_HD
    default: break;
  }
  return MTS_E_UNSUPPORTED;   // not reached: mts_band_attn_bf16_supported lists exactly the instantiations above
}
