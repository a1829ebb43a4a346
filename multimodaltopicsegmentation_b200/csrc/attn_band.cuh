// Pieces shared by the banded-attention kernels on tcgen05 (attn_tc.cu: fp32 q/k/v, attn_bf16.cu: bf16 q/k/v): tile
// shapes, the persistent CTA's walk over work items (Seq / Item / Cursor), tensor-memory and shared-memory access helpers.
#pragma once
#include <cuda.h>

#include "tcgen05_utils.cuh"

namespace mts {
namespace atc {

constexpr int BQ = 128, KT = 64;
constexpr int WORKERS = 256;               // 8 uniform worker warps
constexpr int THREADS = 12 * 32;           // + warp 8 (MMA issuer); warps 9-11 idle (registers are allocated per 4 warps)
constexpr int META_B = 512;                // episodes whose (length, offset) are cached in shared memory
constexpr int TRS = 20;  // floats per row of a per-warp 32 x 16 transposition buffer (80 B: 16-byte aligned rows)
constexpr float LOG2E = 1.4426950408889634f;
constexpr float RESCALE_TH = 5.5f;  // the reference maximum of a row moves only when a tile's maximum exceeds it by this much

// MN-major SWIZZLE_128B descriptor (16-bit operands): LBO = byte stride between 128-byte chunks along N, SBO = between
// groups of 8 K rows (cute/atom/mma_traits_sm100.hpp: ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units)
__device__ __forceinline__ uint64_t desc_sw128_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
constexpr uint32_t B_MN_MAJOR = 1u << 16;  // instruction descriptor: B operand is MN-major

__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, float *v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, float *v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t *v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
      "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ int lds_i32(uint32_t addr) {
  int v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ float4 lds128f(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts128f(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 f4_bits(float4 v) {
  return make_uint4(__float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w));
}
__device__ __forceinline__ uint4 bf16x8(float4 a, float4 b) {
  return make_uint4(bf16x2_bits(a.x, a.y), bf16x2_bits(a.z, a.w), bf16x2_bits(b.x, b.y), bf16x2_bits(b.z, b.w));
}
__device__ __forceinline__ float4 rest4(float4 v) {
  return make_float4(tf32_rest_exact(v.x), tf32_rest_exact(v.y), tf32_rest_exact(v.z), tf32_rest_exact(v.w));
}

// mbarrier wait with the watchdog of tc::bar_wait_wd (a protocol error traps instead of hanging the GPU).  Inline: an
// out-of-line spin makes every wait a call site, and the ~150 live registers of a worker get saved around each.
__device__ __forceinline__ void bar_wait(uint32_t bar, uint32_t parity) { tc::bar_wait_wd(bar, parity); }

// The sequence of work items of a CTA: item = (episode b, query block qb, head), head fastest; CTA c takes items c, c + step, ...
struct Seq {
  int nheads, n_qb, S, w, n_items, step;
  int s_head, s_qb, s_b;   // step decomposed: step = (s_b * n_qb + s_qb) * nheads + s_head
  const int32_t *lengths, *offsets;
  uint32_t meta;           // shared-memory copy of (lengths, offsets) of the first META_B episodes: a global load per look-up
                           // would put an L2 round trip on every step of the tile cursors
};
// one work item, as every role derives it (same arithmetic everywhere keeps the roles' barrier phases in step)
struct Item {
  int idx, b, qb, head;    // position in the sequence
  int q0, len, Sq, kbeg, kend, nt;
  int64_t row0;
  bool active;
};
__device__ __forceinline__ void item_fill(Item &it, const Seq &sq) {
  it.q0 = it.qb * BQ;
  it.active = false;
  it.nt = 0;
  if (it.idx >= sq.n_items) return;
  const bool cached = it.b < META_B;
  it.len = min(max(cached ? lds_i32(sq.meta + 4 * it.b) : __ldg(sq.lengths + it.b), 0), sq.S);
  // ragged layout (offsets != NULL): episode b owns rows offsets[b] .. offsets[b] + len - 1 and nothing beyond
  it.row0 = sq.offsets ? (int64_t)(cached ? lds_i32(sq.meta + 4 * (META_B + it.b)) : __ldg(sq.offsets + it.b)) : (int64_t)it.b * sq.S;
  it.Sq = sq.offsets ? it.len : sq.S;
  it.active = it.q0 < it.len;
  it.kbeg = max(0, it.q0 - sq.w);
  it.kend = min(it.len, it.q0 + BQ + sq.w);
  it.nt = it.active ? (it.kend - it.kbeg + KT - 1) / KT : 0;
}
__device__ __forceinline__ void item_first(Item &it, const Seq &sq, int start) {
  it.idx = start;
  it.head = start % sq.nheads;
  const int rest = start / sq.nheads;
  it.qb = rest % sq.n_qb;
  it.b = rest / sq.n_qb;
  item_fill(it, sq);
}
__device__ __forceinline__ void item_step(Item &it, const Seq &sq) {   // the CTA's next item (active or not)
  it.idx += sq.step;
  it.head += sq.s_head;
  int c = it.head >= sq.nheads;
  it.head -= c ? sq.nheads : 0;
  it.qb += sq.s_qb + c;
  c = it.qb >= sq.n_qb;
  it.qb -= c ? sq.n_qb : 0;
  it.b += sq.s_b + c;
  item_fill(it, sq);
}
// position in a CTA's sequence of key tiles (item-major): active item + tile inside it; valid = not past the end
struct Cursor {
  Item it;
  int t;
  bool valid;
};
__device__ __forceinline__ void cursor_settle(Cursor &c, const Seq &sq) {   // skip inactive items
  while (c.it.idx < sq.n_items && !c.it.active) item_step(c.it, sq);
  c.t = 0;
  c.valid = c.it.idx < sq.n_items;
}
__device__ __forceinline__ void cursor_first(Cursor &c, const Seq &sq, int start) {
  item_first(c.it, sq, start);
  cursor_settle(c, sq);
}
__device__ __forceinline__ void cursor_advance(Cursor &c, const Seq &sq) {   // next key tile (possibly the next active item's first)
  if (++c.t < c.it.nt) return;
  item_step(c.it, sq);
  cursor_settle(c, sq);
}

// descriptor = (constant upper word, lower word = (address >> 4) | LBO << 16): stepping through an operand only adds to the
// lower word
__device__ __forceinline__ uint64_t desc_add(uint64_t base, uint32_t byte_off) { return base + (uint64_t)(byte_off >> 4); }

// First key of tile t of an item.  The raw K / V tiles arrive by TMA as full 64-row boxes; the box of the last tile is shifted
// up so that it ENDS at kend -- it never reads a row behind the episode (behind the buffer, for the last episode of the
// ragged layout).  Rows it re-reads (keys already covered by the previous tile, or -- negative coordinates, zero-filled --
// rows before the buffer) are masked like every other key outside the band.
__device__ __forceinline__ int tile_k0(const Item &it, int t) { return min(it.kbeg + t * KT, it.kend - KT); }

__device__ __forceinline__ void pair_sync(int q) { asm volatile("bar.sync %0, 64;" ::"r"(q + 1) : "memory"); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

}  // namespace atc
}  // namespace mts
