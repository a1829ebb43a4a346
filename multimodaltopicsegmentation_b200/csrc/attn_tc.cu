// Banded (windowed) self-attention, forward, on the 5th-generation tensor cores.
// Same contract as band_attn_fwd_kernel (xfmr.cu): what the reference obtains from HF LongformerSelfAttention
// (models/RestrictedTransformerLayer.py:131 -> HF modeling_longformer.py:481-639, sliding chunks :758-867):
//   softmax over |i - j| <= w, j < len_b of (q_i / sqrt(hd)) . k_j in fp32, exact zeros for padded queries (:578).
//
// One work item = 128 queries of one head of one episode; a persistent CTA per SM walks the items.  Only the key
// tiles (64 keys) intersecting [q0 - w, q0 + 128 + w) x [0, len_b) are read.  Both contractions run as tcgen05.mma
// with the error-compensated operand scheme of the GEMM (common.cuh): x = hi + rest, hi = what kind::tf32 reads of
// the raw fp32 word,
//     S   = Q K^T  ~= hi(Q) hi(K)^T [kind::tf32]  +  bf16(Q) bf16(rest K)^T + bf16(rest Q) bf16(K)^T [kind::f16, packed]
//     O  += P V    ~= hi(P) hi(V)   [kind::tf32]  +  bf16(P) bf16(rest V)   + bf16(rest P) bf16(V)   [kind::f16, packed]
// i.e. fp32-grade scores and outputs (relative error ~2^-19 per product).  The packed correction operands are
// derived ON CHIP from the raw fp32 rows (nothing but q, k, v is read from HBM, nothing but o written).
//
// Tensor memory (512 columns):  Q raw fp32 [0,HD)  (A operand of S, .ts form)
//                               S / P tiles [128,192) [192,256): the accumulator of Q K^T, overwritten IN PLACE by
//                                  the raw fp32 probabilities = the A operand of P V
//                               packed bf16 correction operand of P [256,320) [320,384)
//                               O accumulator [384, 384+HD), accumulated over the key tiles of an item
// Shared memory: packed correction operand of Q (K-major SWIZZLE_128B planes of 32 head columns), the K tile (raw +
//   packed correction, K-major: N = keys, K = head dim) and the V tile (raw + packed correction, MN-major: N = head
//   dim, K = keys; tf32 MN-major operands exist in the SWIZZLE_128B_BASE32B layout only).
//
// Warps: 8 UNIFORM worker warps + 1 MMA-issuing warp + 2 loader warps (one thread each: TMA requests for the raw K / V tiles).  (A first version gave every job its own warps -- softmax, rescale,
// loaders -- with one warp per scheduler and job: correct, but bound by instruction fetch at 0.2 IPC, ncu: 2.5 stalled
// "no instruction" warp-cycles per issued instruction, instruction-cache hit rate 65-72 %.  Now all CUDA-core work is
// done by the same eight warps running the same code, phase after phase, two warps per scheduler.)
//   worker warp w: TMEM lane quarter q = w & 3 (rows 32 q .. 32 q + 31), column half ch = w >> 2.  Per key tile, in order:
//     1. operands of the NEXT tile's S: (new item: Q rows -> tensor memory + packed correction -> shared memory,
//        coalesced loads transposed through shared memory;) K tile: global -> registers (prefetched one tile ahead)
//        -> raw plane + packed correction plane; fence.proxy.async; mbarrier.  The MMA warp then issues S_{t+1}.
//     2. softmax of tile t on my 32 rows x 32 columns: tcgen05.ld S, band / length mask, partial row maxima exchanged
//        with the partner warp through shared memory, p = 2^((s - m) log2 e), tcgen05.st P (raw + packed correction).
//        The reference maximum of a row only moves when a tile exceeds it by RESCALE_TH (p <= e^TH, harmless in fp32),
//        so the rescale O *= alpha (tcgen05.ld / st) is rare.  16-key blocks outside the band of the warp's rows are skipped.
//     3. V tile of tile t: registers -> raw plane + packed correction plane.  The MMA warp then issues O += P V.
//   After the last tile: o / l transposed through shared memory, row-contiguous stores of o (+ the packed correction
//   operand the next GEMM wants) and the log-sum-exp.
//   The tensor pipe works on S_{t+1} during the softmax of tile t and on P V of tile t during the next tile's phase 1.
#include <stdlib.h>

#include "attn_band.cuh"

namespace mts {
namespace atc {

constexpr uint32_t COL_Q = 0, COL_S = 128, COL_PC = 256, COL_O = 384;

template <int HD>
struct Cfg {
  static_assert(HD % 16 == 0 && HD >= 16 && HD <= 128, "head dim: multiple of 16, at most 128");
  static constexpr int NP = (HD + 31) / 32;   // 32-column planes of a raw fp32 / packed-correction operand
  static constexpr int NPV = (HD + 63) / 64;  // 64-column planes of the MN-major bf16 correction operand of V
  static constexpr int C8 = HD / 8;           // 8-float units per row
  static constexpr int NC = HD / 16;          // 16-column chunks per row
  static constexpr int QC_BYTES = NP * BQ * 128;
  static constexpr int KH_BYTES = NP * KT * 128;
  static constexpr int VC_BYTES = NPV * 2 * KT * 128;
  static constexpr int OFF_QC = 0;
  static constexpr int OFF_KH = OFF_QC + QC_BYTES;
  static constexpr int OFF_KC = OFF_KH + KH_BYTES;
  static constexpr int OFF_VH = OFF_KC + KH_BYTES;
  static constexpr int OFF_VC = OFF_VH + KH_BYTES;
  static constexpr int OFF_TR = OFF_VC + VC_BYTES;
  static constexpr int TR_BYTES = 8 * 32 * TRS * 4;
  static constexpr int OFF_MX = OFF_TR + TR_BYTES;           // [2 tile parity][2 column halves][128] partial row maxima
  static constexpr int OFF_LS = OFF_MX + 2 * 2 * BQ * 4;     // [2 column halves][128] partial row sums
  static constexpr int OFF_BAR = OFF_LS + 2 * BQ * 4;
  static constexpr int OFF_META = OFF_BAR + 16 * 8 + 16;     // [2][META_B] int32: lengths, offsets of the first META_B episodes
  static constexpr int USED = OFF_META + 2 * META_B * 4;
  // every CTA allocates all 512 TMEM columns, so two CTAs must never share an SM: ask for more than half its shared memory
  static constexpr int SMEM = (USED + 1024) > 120 * 1024 ? (USED + 1024) : 120 * 1024;
};

enum { B_QREADY = 0, B_QFREE, B_KFULL, B_KEMPTY, B_VFULL, B_VEMPTY, B_SFULL0, B_SFULL1, B_PREADY0, B_PREADY1, B_ODONE, B_OFREE,
       B_KRAW, B_VRAW, B_COUNT };
static_assert(B_COUNT <= 16, "barrier block holds 16 mbarriers");

// MN-major 32-bit (tf32) operands only exist in the SWIZZLE_128B_BASE32B layout (layout type 1, Swizzle<2,5,2> on the byte
// address: the 32-byte unit index, bits 5-6, is XORed with the K row index, bits 7-8): atoms of 4 K rows x 128 bytes
// (32 fp32 along N), SBO = byte stride between groups of 4 K rows, LBO = between 128-byte chunks along N.
__device__ __forceinline__ uint64_t desc_sw128b32_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;
  return d;
}

// Optional in-kernel timeline (off unless mts_debug_attn_profile() installs a buffer): CTA 0 stamps clock64() at the phase
// boundaries of its first AP_ITEMS active items -- role 0 = worker thread 0, role 4 = the MMA thread.
constexpr int AP_ITEMS = 6, AP_ROLES = 5, AP_SLOTS = 40;
__device__ long long *g_atc_prof = nullptr;
#ifdef MTS_ATTN_TIMELINE
#define AP_STAMP(role, slot)                                                                                     \
  do {                                                                                                           \
    if (prof && item_g < (uint32_t)AP_ITEMS && (slot) < AP_SLOTS)                                                \
      prof[((int)item_g * AP_ROLES + (role)) * AP_SLOTS + (slot)] = clock64();                                    \
  } while (0)
#else
#define AP_STAMP(role, slot) \
  do {                       \
    (void)prof;              \
  } while (0)
#endif


// S = Q K^T of one key tile: HD / 8 kind::tf32 MMAs (A = raw Q rows in tensor memory, B = raw K tile) + HD / 8 kind::f16
// MMAs over the packed correction operands.  Called by the whole MMA warp; one elected lane issues.  ONE copy in the
// instruction stream (the role code of five roles shares the instruction cache).
template <int HD>
__device__ __noinline__ void issue_qk(bool leader, uint32_t d_s, uint32_t q_tmem, uint64_t kh_desc, uint64_t qc_desc, uint64_t kc_desc) {
  constexpr uint32_t id_s = tc::idesc_tf32(BQ, KT), id_sc = tc::idesc_bf16(BQ, KT);
#pragma unroll
  for (int ks = 0; ks < HD / 8; ++ks) {
    const uint64_t bd = desc_add(kh_desc, (uint32_t)((ks >> 2) * (KT * 128) + (ks & 3) * 32));
    if (leader) tc::umma_tf32_ts(d_s, q_tmem + 8 * ks, bd, id_s, ks != 0);
  }
#pragma unroll
  for (int j = 0; j < HD / 8; ++j) {
    const uint64_t ad = desc_add(qc_desc, (uint32_t)((j >> 2) * (BQ * 128) + (j & 3) * 32));
    const uint64_t bd = desc_add(kc_desc, (uint32_t)((j >> 2) * (KT * 128) + (j & 3) * 32));
    if (leader) tc::umma_bf16_ss(d_s, ad, bd, id_sc, 1);
  }
}


// Packed correction plane of a K / V tile from its raw plane (both in shared memory; the raw plane arrived by TMA).
// Worker warp wk takes rows 8 wk .. 8 wk + 7; lane = 16-byte piece p of a row (HD / 4 pieces; 32 / (HD / 4) rows per pass).
//   raw plane     K (K-major, SWIZZLE_128B): 16-byte chunk (p & 7) XOR (row & 7) of plane p >> 3
//                 V (MN-major tf32, SWIZZLE_128B_BASE32B = TMA's 128B_ATOM_32B): 32-byte unit ((p >> 1) & 3) XOR (row & 3), half p & 1
//   correction    K (K-major packed, B side: per 16 columns [bf16(rest) x16 | bf16(x) x16]): 8 bytes at 8 (p & 3) of the
//                   rest half / the x half of 64-byte block (p >> 2) & 1 of plane p >> 3
//                 V (MN-major packed: K' rows per 16 keys [rest v x16 | v x16], 64 head columns per 128-byte row): 8 bytes at
//                   column byte 8 (p & 15) of K' row (key >> 4) * 32 + (key & 15) (+ 16 for the v half), plane p >> 4
template <int HD, bool IS_V>
__device__ __forceinline__ void tile_correction(uint32_t hi_base, uint32_t co_base, int wk, int lane) {
  constexpr int LPR = HD / 4, RPI = 32 / LPR > 0 ? 32 / LPR : 1, NI = 8 / RPI;
  const int rsub = lane / LPR, p = lane % LPR;
  if (rsub >= RPI) return;
  uint4 raw[NI];
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int row = 8 * wk + i * RPI + rsub;
    const uint32_t prow = hi_base + (uint32_t)((p >> 3) * (KT * 128) + row * 128);
    raw[i] = lds128(prow + (uint32_t)(IS_V ? (((((p >> 1) & 3) ^ (row & 3)) << 5) + 16 * (p & 1)) : (((p & 7) ^ (row & 7)) << 4)));
  }
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int row = 8 * wk + i * RPI + rsub;
    const float4 x = make_float4(__uint_as_float(raw[i].x), __uint_as_float(raw[i].y), __uint_as_float(raw[i].z), __uint_as_float(raw[i].w));
    const uint2 xb = make_uint2(bf16x2_bits(x.x, x.y), bf16x2_bits(x.z, x.w));
    const uint2 rb = make_uint2(bf16x2_bits(tf32_rest_exact(x.x), tf32_rest_exact(x.y)),
                                bf16x2_bits(tf32_rest_exact(x.z), tf32_rest_exact(x.w)));
    if (!IS_V) {
      const uint32_t prow = co_base + (uint32_t)((p >> 3) * (KT * 128) + row * 128);
      const int chunk = ((p >> 2) & 1) * 4 + ((p & 3) >> 1);
      asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(prow + (uint32_t)(((chunk ^ (row & 7)) << 4) + 8 * (p & 1))), "r"(rb.x), "r"(rb.y) : "memory");
      asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(prow + (uint32_t)((((chunk + 2) ^ (row & 7)) << 4) + 8 * (p & 1))), "r"(xb.x), "r"(xb.y) : "memory");
    } else {
      const int rr = (row >> 4) * 32 + (row & 15);
      const uint32_t ca = co_base + (uint32_t)((p >> 4) * (2 * KT * 128) + rr * 128 + (((((p & 15) >> 1)) ^ (rr & 7)) << 4) + 8 * (p & 1));
      asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(ca), "r"(rb.x), "r"(rb.y) : "memory");
      asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(ca + 16 * 128), "r"(xb.x), "r"(xb.y) : "memory");
    }
  }
}

template <int HD>
__global__ void __launch_bounds__(THREADS, 1)
    band_attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v,
                            const float *__restrict__ qkv, int64_t ld, const int32_t *__restrict__ lengths,
                            const int32_t *__restrict__ offsets, int B, int S, int nheads, int w, float *__restrict__ out,
                            float *__restrict__ out_hi, float *__restrict__ out_lo, int Kp, float *__restrict__ lse) {
  using C = Cfg<HD>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t sbase = tc::s_u32(smem);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + C::OFF_BAR);
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 16);
  int32_t *meta_p = reinterpret_cast<int32_t *>(smem + C::OFF_META);
  const uint32_t mx_s = sbase + C::OFF_MX, ls_s = sbase + C::OFF_LS;

  const int lane = threadIdx.x & 31;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp-uniform for the compiler
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
    tc::bar_init(BAR(B_QREADY), WORKERS);
    tc::bar_init(BAR(B_QFREE), 1);
    tc::bar_init(BAR(B_KFULL), WORKERS);
    tc::bar_init(BAR(B_KEMPTY), 1);
    tc::bar_init(BAR(B_VFULL), WORKERS);
    tc::bar_init(BAR(B_VEMPTY), 1);
    tc::bar_init(BAR(B_SFULL0), 1);
    tc::bar_init(BAR(B_SFULL1), 1);
    tc::bar_init(BAR(B_PREADY0), WORKERS);
    tc::bar_init(BAR(B_PREADY1), WORKERS);
    tc::bar_init(BAR(B_ODONE), 1);
    tc::bar_init(BAR(B_OFREE), WORKERS);
    tc::bar_init(BAR(B_KRAW), 1);
    tc::bar_init(BAR(B_VRAW), 1);
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
    const uint32_t tr = sbase + (uint32_t)(C::OFF_TR + warp * 32 * TRS * 4);   // my warp's transposition buffer (shared-space address:
                                                                             // a generic pointer makes every access a generic LD / ST)
    const float inv_scale = 1.0f / sqrtf((float)HD);   // HF divides q by sqrt(head_dim) (:513); the product differs by <= 1 ulp
    long long *prof = (blockIdx.x == 0 && threadIdx.x == 0) ? g_atc_prof : nullptr;
    uint32_t item_g = 0, tile_g = 0;                 // items / tiles completed (softmax view)
    uint32_t k_cnt = 0, v_cnt = 0, q_cnt = 0;        // K tiles, V tiles, Q blocks handed over so far

    // ck: the next S tile of the sequence whose operands are to be handed over
    Cursor ck;
    cursor_first(ck, sq, blockIdx.x);
    bool started = false;   // the sequence's first tile still needs its S operands (done by a virtual pass t = -1)
    Item it;
    for (item_first(it, sq, blockIdx.x); it.idx < sq.n_items; item_step(it, sq)) {
      float inv = 0.0f, lse_v = 0.0f;
      if (it.active) {
        AP_STAMP(0, 0);
        const int i = it.q0 + r;
        float m_run = -INFINITY, l_run = 0.0f;
#pragma unroll 1
        for (int t = started ? 0 : -1; t < it.nt; ++t) {
          // ---- phase 1: operands of the NEXT S tile of the sequence (its raw K tile arrives by TMA) ----------------------
          if (ck.valid) {
            if (ck.t == 0) {
              // The tile opens a new item: its Q (16-column chunks c = ch, ch + 2, ...).  Coalesced loads (a warp instruction =
              // 8 rows x 64 contiguous bytes), all chunks in flight at once, transposed through the warp's buffer so that
              // every lane holds ITS row; raw fp32 -> tensor memory, packed correction operand (A side: per 16 columns
              // [bf16(x) x16 | bf16(rest) x16]) -> shared memory.
              const Item &qi = ck.it;
              AP_STAMP(0, 20);
              const float *qbase = qkv + qi.row0 * ld + qi.head * HD + 4 * (lane & 3);
              const int rr0 = lane >> 2;
              constexpr int MYC = (C::NC + 1) / 2;
              float4 nx[MYC][4];
              // straight-line, unconditional loads (rows beyond the episode: clamped address, value zeroed by the scale
              // factor below) -- a branch around each load made the compiler put the first use next to it, i.e. one exposed
              // memory latency per load (measured: 12 000 cycles for these 16 loads)
              float sc[4];
              const float *qrow[4];
#pragma unroll
              for (int i2 = 0; i2 < 4; ++i2) {
                const int gi = qi.q0 + q * 32 + rr0 + 8 * i2;
                sc[i2] = gi < qi.Sq ? inv_scale : 0.0f;
                qrow[i2] = qbase + (int64_t)min(gi, qi.Sq - 1) * ld;
              }
#pragma unroll
              for (int k = 0; k < MYC; ++k) {
                const int c = min(ch + 2 * k, C::NC - 1);   // (an odd chunk count: the last slot of column half 1 re-reads, unused)
#pragma unroll
                for (int i2 = 0; i2 < 4; ++i2) nx[k][i2] = __ldg(reinterpret_cast<const float4 *>(qrow[i2] + 16 * c));
              }
              AP_STAMP(0, 21);
              bar_wait(BAR(B_QFREE), (q_cnt & 1) ^ 1);   // every S = Q K^T of the previous item has completed
              tc::tc_fence_after();
              AP_STAMP(0, 22);
#pragma unroll
              for (int k = 0; k < MYC; ++k) {
                const int c = ch + 2 * k;
                if (c >= C::NC) break;
#pragma unroll
                for (int i2 = 0; i2 < 4; ++i2)
                  sts128f(tr + 4 * ((rr0 + 8 * i2) * TRS + 4 * (lane & 3)),
                          make_float4(nx[k][i2].x * sc[i2], nx[k][i2].y * sc[i2], nx[k][i2].z * sc[i2], nx[k][i2].w * sc[i2]));
                __syncwarp();
                float4 x[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) x[j] = lds128f(tr + 4 * (lane * TRS + 4 * j));
                __syncwarp();
                uint32_t raw[16];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  raw[4 * j] = __float_as_uint(x[j].x); raw[4 * j + 1] = __float_as_uint(x[j].y);
                  raw[4 * j + 2] = __float_as_uint(x[j].z); raw[4 * j + 3] = __float_as_uint(x[j].w);
                }
                tmem_st16(trow + COL_Q + 16 * c, raw);
                const uint32_t rowa = sbase + C::OFF_QC + (uint32_t)((c >> 1) * (BQ * 128) + r * 128);
                const int cb = (c & 1) * 4, sw = r & 7;
                sts128(rowa + (((cb + 0) ^ sw) << 4), bf16x8(x[0], x[1]));
                sts128(rowa + (((cb + 1) ^ sw) << 4), bf16x8(x[2], x[3]));
                sts128(rowa + (((cb + 2) ^ sw) << 4), bf16x8(rest4(x[0]), rest4(x[1])));
                sts128(rowa + (((cb + 3) ^ sw) << 4), bf16x8(rest4(x[2]), rest4(x[3])));
              }
              AP_STAMP(0, 23);
              tc::tmem_wait_st();
              tc::fence_proxy_async();
              tc::tc_fence_before();
              tc::bar_arrive(BAR(B_QREADY));
              AP_STAMP(0, 24);
              ++q_cnt;
            }
            bar_wait(BAR(B_KRAW), k_cnt & 1);   // the raw K tile has landed (requested by the loader warp when its buffer fell free)
            AP_STAMP(0, 25);
            tile_correction<HD, false>(sbase + C::OFF_KH, sbase + C::OFF_KC, warp, lane);
            tc::fence_proxy_async();
            tc::bar_arrive(BAR(B_KFULL));
            AP_STAMP(0, 26);
            ++k_cnt;
            cursor_advance(ck, sq);
          }
          if (t < 0) {   // virtual pass: only the operands of the sequence's first S tile
            started = true;
            continue;
          }
          AP_STAMP(0, 1 + 4 * t);
          // ---- phase 2: softmax of tile t, my 32 rows x 32 columns -------------------------------------------------------
          const int buf = tile_g & 1;
          const int k0 = tile_k0(it, t) + 32 * ch;     // first key of my column half
          // valid column range [clo, clo + nvalid) of my row inside my half: band |i - j| <= w, j < kend (<= len), and not a
          // key the previous tile has covered already (the last tile's box is shifted up to end at kend)
          const int clo = max(max(0, i - w - k0), it.kbeg + t * KT - k0);
          const int chi = (i < it.len) ? min(it.kend - k0, i + w + 1 - k0) : 0;
          const unsigned nvalid = (unsigned)max(min(chi, 32) - clo, 0);
          bar_wait(BAR(B_SFULL0 + buf), (tile_g >> 1) & 1);
          tc::tc_fence_after();
          AP_STAMP(0, 2 + 4 * t);
          float s[32];
          tmem_ld32_nowait(trow + COL_S + 64 * buf + 32 * ch, s);
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
              s[c] = ((unsigned)(c - clo) < nvalid) ? s[c] : -INFINITY;
              mx4[e & 3] = fmaxf(mx4[e & 3], s[c]);
            }
          }
          // row maximum over both column halves: exchange with the partner warp
          float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
          sts_f32(mx_s + 4 * ((buf * 2 + ch) * BQ + r), mx);
          pair_sync(q);
          mx = fmaxf(mx, lds_f32(mx_s + 4 * ((buf * 2 + (ch ^ 1)) * BQ + r)));
          // reference maximum: moved only when this tile exceeds it by more than RESCALE_TH (first valid tile: always)
          float alpha = 1.0f;
          if (mx > m_run + RESCALE_TH) {   // false while mx == -inf; true for the first finite mx (m_run == -inf)
            if (m_run != -INFINITY) { alpha = ex2f((m_run - mx) * LOG2E); l_run *= alpha; }
            m_run = mx;
          }
          if (t > 0 && __any_sync(0xffffffffu, alpha != 1.0f)) {
            // rare: rescale my column half of O (16-column chunks c = ch, ch + 2, ...); the previous P V must be complete
            bar_wait(BAR(B_VEMPTY), (v_cnt & 1) ^ 1);
            tc::tc_fence_after();
#pragma unroll 1
            for (int c = ch; c < C::NC; c += 2) {
              float v[16];
              uint32_t u[16];
              tmem_ld16_nowait(trow + COL_O + 16 * c, v);
              tmem_wait_ld();
#pragma unroll
              for (int e = 0; e < 16; ++e) u[e] = __float_as_uint(v[e] * alpha);
              tmem_st16(trow + COL_O + 16 * c, u);
            }
          }
          const float mb = (m_run == -INFINITY) ? 0.0f : -m_run * LOG2E;
          float ps4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
          for (int blk = 0; blk < 2; ++blk) {
            uint32_t ph[16], pc[16];
            if (live & (1u << blk)) {
#pragma unroll
              for (int e = 0; e < 16; e += 2) {
                const float p0 = ex2f(fmaf(s[16 * blk + e], LOG2E, mb)), p1 = ex2f(fmaf(s[16 * blk + e + 1], LOG2E, mb));
                ps4[(e >> 1) & 3] += p0 + p1;
                ph[e] = __float_as_uint(p0);
                ph[e + 1] = __float_as_uint(p1);
                pc[e >> 1] = bf16x2_bits(p0, p1);
                pc[8 + (e >> 1)] = bf16x2_bits(tf32_rest_exact(p0), tf32_rest_exact(p1));
              }
            } else {
#pragma unroll
              for (int e = 0; e < 16; ++e) ph[e] = pc[e] = 0u;
            }
            tmem_st16(trow + COL_S + 64 * buf + 32 * ch + 16 * blk, ph);    // raw fp32 probabilities, in place of the scores
            tmem_st16(trow + COL_PC + 64 * buf + 32 * ch + 16 * blk, pc);   // [bf16(p) x16 | bf16(rest p) x16]
          }
          l_run += (ps4[0] + ps4[1]) + (ps4[2] + ps4[3]);
          tc::tmem_wait_st();
          tc::tc_fence_before();
          tc::bar_arrive(BAR(B_PREADY0 + buf));
          AP_STAMP(0, 3 + 4 * t);
          // ---- phase 3: V tile of tile t (prefetched), then prefetch the next V tile of the sequence --------------------
          bar_wait(BAR(B_VRAW), v_cnt & 1);   // the raw V tile has landed
          tile_correction<HD, true>(sbase + C::OFF_VH, sbase + C::OFF_VC, warp, lane);
          tc::fence_proxy_async();
          tc::bar_arrive(BAR(B_VFULL));
          ++v_cnt;
          ++tile_g;
          AP_STAMP(0, 4 + 4 * t);
        }
        // row sums of the two column halves
        sts_f32(ls_s + 4 * (ch * BQ + r), l_run);
        pair_sync(q);
        const float l_tot = l_run + lds_f32(ls_s + 4 * ((ch ^ 1) * BQ + r));
        const bool alive = (i < it.len) && (l_tot > 0.0f);
        inv = alive ? 1.0f / l_tot : 0.0f;
        lse_v = alive ? m_run + logf(l_tot) : 0.0f;
        pair_sync(q);   // ls_s may be rewritten by the next item only after both have read
        bar_wait(BAR(B_ODONE), item_g & 1);   // the last P V of the item has completed
        tc::tc_fence_after();
        AP_STAMP(0, 38);
      }
      // ---- o / l, transposed through the warp's buffer, row-contiguous stores (+ the next GEMM's correction operand) ----
      // (inactive item = a block of padded queries: exact zeros, HF :578; nothing exists there in the ragged layout)
      if (it.q0 < it.Sq) {
#pragma unroll 1
        for (int c = ch; c < C::NC; c += 2) {
          float v[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) v[e] = 0.0f;
          if (it.active) {
            tmem_ld16_nowait(trow + COL_O + 16 * c, v);
            tmem_wait_ld();
          }
#pragma unroll
          for (int j = 0; j < 4; ++j)
            sts128f(tr + 4 * (lane * TRS + 4 * j), make_float4(v[4 * j] * inv, v[4 * j + 1] * inv, v[4 * j + 2] * inv, v[4 * j + 3] * inv));
          __syncwarp();
          // a warp instruction = 8 rows x 64 contiguous bytes (4 lanes per row): raw values, then the packed correction
          // operand of the 16-column block: [bf16(x) 0-7 | bf16(x) 8-15 | bf16(rest) 0-7 | bf16(rest) 8-15], 16 bytes per lane
#pragma unroll
          for (int i2 = 0; i2 < 4; ++i2) {
            const int rr = (lane >> 2) + 8 * i2, pc4 = lane & 3, gi = it.q0 + q * 32 + rr;
            if (gi < it.Sq) {
              const int col = it.head * HD + 16 * c;
              const float4 a = lds128f(tr + 4 * (rr * TRS + 4 * pc4));
              if (out) *reinterpret_cast<float4 *>(out + (it.row0 + gi) * d + col + 4 * pc4) = a;
              if (out_hi) {
                *reinterpret_cast<float4 *>(out_hi + (it.row0 + gi) * Kp + col + 4 * pc4) = a;
                float4 e0 = lds128f(tr + 4 * (rr * TRS + 8 * (pc4 & 1)));
                float4 e1 = lds128f(tr + 4 * (rr * TRS + 8 * (pc4 & 1) + 4));
                if (pc4 >= 2) { e0 = rest4(e0); e1 = rest4(e1); }
                // the operand row holds 2 Kp bf16 in Kp floats: block (col / 16) starts at float col (= 64 bytes per 16 columns)
                *reinterpret_cast<uint4 *>(out_lo + (it.row0 + gi) * Kp + col + 4 * pc4) = bf16x8(e0, e1);
              }
            }
          }
          __syncwarp();
        }
      }
      if (it.active) {
        tc::tc_fence_before();
        tc::bar_arrive(BAR(B_OFREE));   // my reads of O are done: the next item's first P V may overwrite it
        AP_STAMP(0, 39);
        ++item_g;
      }
      if (ch == 0 && lse && it.q0 + r < S) lse[((int64_t)it.b * nheads + it.head) * S + it.q0 + r] = lse_v;
    }
  } else if (warp == 9 || warp == 10) {
    // =============================== loader warps: raw K (warp 9) / V (warp 10) tiles by TMA ===============================
    // One request per tile as soon as its buffer falls free (the S / P V product that read the previous tile has completed),
    // i.e. a whole softmax phase before the workers need it: 64 rows x 32 columns per plane, swizzled by the TMA unit the way
    // the tensor core wants the operand.
    if (lane == 0) {
      const bool is_v = warp == 10;
      const CUtensorMap *map = is_v ? &map_v : &map_k;
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
      const uint32_t dst = sbase + (uint32_t)(is_v ? C::OFF_VH : C::OFF_KH);
      const uint32_t raw_bar = BAR(is_v ? B_VRAW : B_KRAW), empty_bar = BAR(is_v ? B_VEMPTY : B_KEMPTY);
      Cursor cl;
      uint32_t n = 0;
      for (cursor_first(cl, sq, blockIdx.x); cl.valid; cursor_advance(cl, sq), ++n) {
        bar_wait(empty_bar, (n & 1) ^ 1);
        tc::bar_expect_tx(raw_bar, C::NP * KT * 128);
        const int c0 = (is_v ? 2 : 1) * d + cl.it.head * HD, c1 = (int)cl.it.row0 + tile_k0(cl.it, cl.t);
#pragma unroll
        for (int j = 0; j < C::NP; ++j) tma_load_2d(dst + j * (KT * 128), map, c0 + 32 * j, c1, raw_bar);
      }
    }
  } else if (warp == 8) {
    // =============================== MMA issuer: warp-uniform control flow, one elected lane ===============================
    constexpr uint32_t id_o = tc::idesc_tf32(BQ, HD) | B_MN_MAJOR, id_oc = tc::idesc_bf16(BQ, HD) | B_MN_MAJOR;
    const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
    const bool leader = tc::elect_one();
    const uint64_t kh_desc = tc::desc_sw128(sbase + C::OFF_KH), qc_desc = tc::desc_sw128(sbase + C::OFF_QC);
    const uint64_t kc_desc = tc::desc_sw128(sbase + C::OFF_KC);
    const uint64_t vh_desc = desc_sw128b32_mn(sbase + C::OFF_VH, KT * 128), vc_desc = desc_sw128_mn(sbase + C::OFF_VC, 2 * KT * 128);
    uint32_t item_g = 0, tile_g = 0, s_cnt = 0, q_seen = 0;
    long long *prof = (blockIdx.x == 0 && lane == 0) ? g_atc_prof : nullptr;

    // cs: the next S tile to issue (kept one ahead of the P V position cp)
    Cursor cs, cp;
    cursor_first(cs, sq, blockIdx.x);
    cp = cs;
    bool started = false;
    while (cp.valid) {
      const int nt = cp.it.nt;
#pragma unroll 1
      for (int t = started ? 0 : -1; t < nt; ++t) {
        if (cs.valid) {
          // S = Q K^T of the sequence's next tile: one ahead of the softmax
          if (cs.t == 0) {   // the tile opens a new item: its Q must have landed
            bar_wait(BAR(B_QREADY), q_seen & 1);
            ++q_seen;
          }
          const uint32_t sbuf = s_cnt & 1;
          bar_wait(BAR(B_KRAW), s_cnt & 1);    // (complete by now; orders the TMA writes before this thread's MMAs)
          bar_wait(BAR(B_KFULL), s_cnt & 1);
          tc::tc_fence_after();
          AP_STAMP(4, 1 + 4 * (t + 1));
          issue_qk<HD>(leader, tb + COL_S + 64 * sbuf, tb + COL_Q, kh_desc, qc_desc, kc_desc);
          if (leader) {
            tc::umma_commit(BAR(B_SFULL0 + sbuf));
            tc::umma_commit(BAR(B_KEMPTY));
            if (cs.t == cs.it.nt - 1) tc::umma_commit(BAR(B_QFREE));   // the item's last S product
          }
          __syncwarp();
#ifdef MTS_ATTN_TIMELINE   // diagnostic: how long does the S product take to execute?
          AP_STAMP(4, 20 + (t + 1));
          bar_wait(BAR(B_SFULL0 + sbuf), (s_cnt >> 1) & 1);
          AP_STAMP(4, 26 + (t + 1));
#endif
          ++s_cnt;
          cursor_advance(cs, sq);
        }
        if (t < 0) {
          started = true;
          continue;
        }
        const uint32_t buf = tile_g & 1;
        bar_wait(BAR(B_PREADY0 + buf), (tile_g >> 1) & 1);
        AP_STAMP(4, 2 + 4 * t);
        bar_wait(BAR(B_VRAW), tile_g & 1);
        bar_wait(BAR(B_VFULL), tile_g & 1);
        if (t == 0) bar_wait(BAR(B_OFREE), (item_g & 1) ^ 1);   // the previous item's epilogue has read O
        tc::tc_fence_after();
        AP_STAMP(4, 3 + 4 * t);
        const uint32_t d_o = tb + COL_O;
#pragma unroll
        for (int kg = 0; kg < KT / 8; ++kg) {
          const uint64_t bd = desc_add(vh_desc, (uint32_t)(kg * 1024));
          if (leader) tc::umma_tf32_ts(d_o, tb + COL_S + 64 * buf + 8 * kg, bd, id_o, (t | kg) != 0);
        }
#pragma unroll
        for (int j = 0; j < 2 * KT / 16; ++j) {
          const uint64_t bd = desc_add(vc_desc, (uint32_t)(j * 2048));
          if (leader) tc::umma_bf16_ts(d_o, tb + COL_PC + 64 * buf + 8 * j, bd, id_oc, 1);
        }
        if (leader) {
          tc::umma_commit(BAR(B_VEMPTY));
          if (t == nt - 1) tc::umma_commit(BAR(B_ODONE));
        }
        __syncwarp();
#ifdef MTS_ATTN_TIMELINE   // diagnostic: how long does the P V product take to execute?
        AP_STAMP(4, 32 + t);
        bar_wait(BAR(B_VEMPTY), tile_g & 1);
        AP_STAMP(4, 36 + t);
#endif
        ++tile_g;
        AP_STAMP(4, 4 + 4 * t);
      }
      ++item_g;
      // P V position: on to the next active item
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

// qkv as a 2-D fp32 tensor [rows, 3 d] (row stride ld); box = 64 rows x 32 columns = one raw operand plane.  `rows` is an
// upper bound (B * S): by construction no box ends behind its episode (tile_k0), so nothing behind the buffer is read.
static int make_map(CUtensorMap *map, const float *qkv, int64_t ld, int width, int64_t rows, CUtensorMapSwizzle swz) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { set_error("band_attn_fwd_tc: cuTensorMapEncodeTiled not available"); return MTS_E_NODEVICE; }
  cuuint64_t dims[2] = {(cuuint64_t)width, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
  cuuint32_t box[2] = {32, (cuuint32_t)KT};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void *)qkv, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("band_attn_fwd_tc: cuTensorMapEncodeTiled failed"); return MTS_E_BADARG; }
  return 0;
}

template <int HD>
static int launch(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B, int S, int nheads, int w,
                  float *out, float *out_hi, float *out_lo, int Kp, float *lse, cudaStream_t st) {
  using C = Cfg<HD>;
  CUtensorMap map_k, map_v;
  int rc;
  if ((rc = make_map(&map_k, qkv, ld, 3 * nheads * HD, (int64_t)B * S, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map(&map_v, qkv, ld, 3 * nheads * HD, (int64_t)B * S, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B))) return rc;
  MTS_CUDA(cudaFuncSetAttribute(band_attn_fwd_tc_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
  const int n_items = B * ((S + BQ - 1) / BQ) * nheads;
  const int grid = n_items < kNumSMs ? n_items : kNumSMs;
  band_attn_fwd_tc_kernel<HD><<<grid, THREADS, C::SMEM, st>>>(map_k, map_v, qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi,
                                                             out_lo, Kp, lse);
  MTS_LAUNCH_CHECK();
  return 0;
}

}  // namespace atc
}  // namespace mts

using namespace mts;

// profiling hook: buf = device buffer of AP_ITEMS * AP_ROLES * AP_SLOTS int64 (or NULL to switch the timeline off)
extern "C" int mts_debug_attn_profile(long long *buf) {
  MTS_CUDA(cudaMemcpyToSymbol(atc::g_atc_prof, &buf, sizeof(buf)));
  return 0;
}

extern "C" int mts_band_attn_tc_supported(int hd) { return hd == 16 || hd == 32 || hd == 64 || hd == 112 || hd == 128; }

extern "C" int mts_band_attn_fwd_tc(const float *qkv, int64_t ld, const int32_t *lengths, const int32_t *offsets, int B, int S,
                                    int nheads, int hd, int w, float *out, float *out_hi, float *out_lo, int Kp, float *lse,
                                    void *stream) {
  MTS_REQUIRE(qkv && lengths && (out || out_hi), MTS_E_BADARG, "band_attn_fwd_tc: null pointer");
  MTS_REQUIRE((out_hi == nullptr) == (out_lo == nullptr), MTS_E_BADARG, "band_attn_fwd_tc: hi and lo go together");
  MTS_REQUIRE(B > 0 && S > 0 && nheads > 0 && hd > 0 && w >= 0, MTS_E_BADARG, "band_attn_fwd_tc: bad shape");
  MTS_REQUIRE(ld % 4 == 0 && ld >= 3 * nheads * hd, MTS_E_BADARG, "band_attn_fwd_tc: qkv row stride");
  MTS_REQUIRE(((uintptr_t)qkv & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)out_hi & 15) == 0 && ((uintptr_t)out_lo & 15) == 0,
              MTS_E_BADARG, "band_attn_fwd_tc: buffers must be 16-byte aligned");
  MTS_REQUIRE(!out_hi || Kp == nheads * hd, MTS_E_UNSUPPORTED, "band_attn_fwd_tc: the split output needs Kp == model width");
  cudaStream_t st = (cudaStream_t)stream;
  switch (hd) {
    case 16: return atc::launch<16>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    case 32: return atc::launch<32>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    case 64: return atc::launch<64>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    case 112: return atc::launch<112>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    case 128: return atc::launch<128>(qkv, ld, lengths, offsets, B, S, nheads, w, out, out_hi, out_lo, Kp, lse, st);
    default: break;
  }
  set_error("band_attn_fwd_tc: head dim must be one of 16, 32, 64, 112, 128");
  return MTS_E_UNSUPPORTED;
}
