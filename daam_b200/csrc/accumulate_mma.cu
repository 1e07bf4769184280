// Fused softmax(QK^T) -> unravel -> accumulate, tcgen05 / TMA / TMEM variant (head_dim up to 192 in 64-wide K chunks).
//
// One tile = 128 pixels x 77 tokens of one (layer, prompt, head). Per tile:
//   TMA        Q tile [128 x 64] and K [77(+3 zero rows) x 64] -> shared memory, 128B-swizzled K-major (the UMMA
//              canonical layout), straight from the strided `to_q`/`to_k` outputs via 4-D tensor maps
//              {dim, head, row, prompt}; partial tiles and the 3 padding token rows are zero-filled by the TMA unit.
//   tcgen05    S = Q K^T as 4 x tcgen05.mma (M128 N80 K16, kind::f16, fp32 accumulate) into a TMEM accumulator
//              (2 accumulators, so the MMA of tile i+1 overlaps the epilogue of tile i).
//   epilogue   4 warps: tcgen05.ld gives every thread the 77 logits of ITS pixel (TMEM lane == pixel), so the
//              softmax is thread-local (no shuffles); the probabilities are then added into the fp32 accumulator
//              acc[head][token][pixel] either
//                red mode : staged token-major in shared memory and sent as ONE bulk-tensor reduce-add
//                           (cp.reduce.async.bulk.tensor .add.f32): the read-modify-write happens in L2, the SM never
//                           loads the accumulator;
//                ldst mode: coalesced 128-byte load / add / store per warp and token, straight from registers.
// Warp roles: 0-3 epilogue, 4 TMA producer (one elected thread), 5 TMEM allocator + MMA issuer (one thread).
// Persistent: CTA b of a grid of G takes the launch's tiles b, b + G, b + 2G, ... (K-chunked launches: a contiguous range
// of equal weight); up to 2 CTAs per SM (256 TMEM columns each).
//
// fp32 projections (the reference's default dtype for SD-1.x/2.x, daam/run/generate.py:205) take the same kernel in
// "split" form. Tensor cores have no fp32 operand type and a plain kind::tf32 product would drop 13 mantissa bits, so
// every value is used as two tf32 terms, x = hi + lo with hi = trunc_tf32(x) -- what the tensor core reads from the raw
// fp32 container -- and lo = rna_tf32(x - hi) (22 significand bits), and q.k = q_lo.k_hi + q_hi.k_lo + q_hi.k_hi (the
// dropped terms are ~2^-22 relative): the fp32 Q/K tiles arrive by TMA exactly like the 16-bit ones (two 128-byte-wide
// swizzled sub-tiles per 64 dims) and ARE the hi operands; eight converter warps emit `lo` into a second buffer (a
// shared-memory -> shared-memory elementwise pass, swizzle-agnostic), and the MMA thread issues 3 x 8 tcgen05.mma
// kind::tf32 (K = 8) per tile. One CTA per SM (two 52 KB raw stages + one lo buffer + the staged probabilities).
//
// head_dim other than 64 (SD-1.x: 40 / 80 / 160): the contraction runs in 64-wide K chunks, one chunk per smem stage,
// accumulated into the same TMEM accumulator; the last chunk is zero-filled beyond head_dim (by the TMA unit, or by the
// converter warps) and issues only the MMAs that cover live columns.
//
// Replaces daam/trace.py:276 (get_attention_scores), :219-244 (_unravel_attn) and :293-294 (update loop).
#include <cuda.h>

#include <mutex>
#include <unordered_map>
#include <string>

#include "common.cuh"

namespace daam {
namespace {

constexpr int kStages = 2;
constexpr int kQBytes = kTilePixels * 128;            // 128 rows x 128 B (64 x 16-bit, or 32 x fp32: one swizzle span)
constexpr int kKBytes = kTokensPad * 128;             // 80 rows x 128 B
constexpr int kStageBytes = kQBytes + kKBytes;        // 26624 = 26 x 1024 (keeps every tile 1024-byte aligned)
constexpr int kPBytes = kTokens * kTilePixels * 4;    // staged probabilities [77][128] fp32
constexpr int kTmemCols = 256;
constexpr int kAccCols = 128;                         // column distance between the two accumulators
constexpr int kThreads = 192;
constexpr int kBarBytes = 256;                        // mbarriers + the TMEM base address slot
constexpr int kSmemBytes = 1024 + kStages * kStageBytes + kPBytes + kBarBytes;
// split (fp32) form: a raw stage holds the fp32 tiles as [Q sub0][Q sub1][K sub0][K sub1] (sub-tile = 32 floats = one
// 128-byte swizzle span per row); one more buffer of the same shape holds the lo terms; warps 6-9 convert
constexpr int kSplitStageBytes = 2 * kStageBytes;     // 53248 = 52 x 1024
constexpr int kSplitThreads = 448;                   // 6 warps as in the 16-bit form + 8 converter warps
constexpr int kSplitSmemBytes = 1024 + (kStages + 1) * kSplitStageBytes + kPBytes + kBarBytes;
static_assert(kSplitSmemBytes <= 232448, "split form exceeds the 227 KB shared-memory limit");

struct MmaParams {
  LaunchParams base;
  CUtensorMap qmap[kMaxLayersPerLaunch];
  CUtensorMap kmap[kMaxLayersPerLaunch];
  CUtensorMap amap[kMaxLayersPerLaunch];
};

// ---- PTX wrappers -------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (reported as a CUDA error) instead of hanging the GPU. The bound is ~10 s of SM
// clocks, far beyond any legitimate wait on a dedicated GPU; where a context can be descheduled for longer (MPS,
// time-slicing, a debugger) build with -DDAAM_MBAR_TIMEOUT_CYCLES=0 to wait without a bound.
#ifndef DAAM_MBAR_TIMEOUT_CYCLES
#define DAAM_MBAR_TIMEOUT_CYCLES 20000000000LL
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try(bar, parity)) return;
#if DAAM_MBAR_TIMEOUT_CYCLES > 0
  const long long t0 = clock64();
  while (!mbar_try(bar, parity)) {
    if (clock64() - t0 > DAAM_MBAR_TIMEOUT_CYCLES) __trap();
  }
#else
  while (!mbar_try(bar, parity)) {}
#endif
}

__device__ __forceinline__ void tma_load_4d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void epi_barrier() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

// UMMA shared-memory descriptor: K-major operand tile, 128B swizzle, rows of 128 bytes, 8-row groups 1024 B apart.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) /* LBO (unused with swizzle) */ |
         ((uint64_t)(1024 >> 4) << 32) /* SBO */ | (1ull << 46) /* descriptor version (sm_100) */ |
         (2ull << 61) /* SWIZZLE_128B */;
}
// Instruction descriptor, kind::f16: fp32 accumulate, A/B both K-major, M = 128, N = 80.
__device__ __forceinline__ uint32_t umma_idesc(bool bf16) {
  const uint32_t fmt = bf16 ? 1u : 0u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(kTokensPad >> 3) << 17) |
         ((uint32_t)(kTilePixels >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::tf32: operands are 32-bit containers read as tf32, K = 8 per instruction (32 bytes along the swizzled row).
__device__ __forceinline__ uint32_t umma_idesc_tf32() {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kTokensPad >> 3) << 17) | ((uint32_t)(kTilePixels >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

struct Tile {
  int li, prompt, head, pixel0;
};
__device__ __forceinline__ Tile decode_tile(const LaunchParams& P, int tile, int& li) {
  while (li + 1 < P.n_layers && tile >= P.layer[li + 1].tile_begin) ++li;
  const LayerParams& L = P.layer[li];
  const int local = tile - L.tile_begin;
  const int ptile = local % L.tiles_per_head;
  const int ph = local / L.tiles_per_head;
  Tile t;
  t.li = li;
  t.head = ph % L.heads;
  t.prompt = ph / L.heads;
  t.pixel0 = ptile * kTilePixels;
  return t;
}

// First tile whose weight offset (tiles before it x their weights) is >= w; total_tiles for w >= total_weight.
__device__ __forceinline__ int tile_at_weight(const LaunchParams& P, long long w) {
  if (w >= P.total_weight) return P.total_tiles;
  int li = 0;
  while (li + 1 < P.n_layers && w >= P.layer[li + 1].weight_begin) ++li;
  const LayerParams& L = P.layer[li];
  return L.tile_begin + (int)((w - L.weight_begin + L.weight - 1) / L.weight);
}

__device__ __forceinline__ float rna_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
// hi term of the split as the tensor core sees it: kind::tf32 reads the upper 19 bits of the 32-bit container and
// ignores the low 13 mantissa bits, i.e. hi = trunc_tf32(x). (Pinned by tests/test_parity_elementwise_gpu.py: were the
// hardware to round instead, hi + lo would be off by a tf32 ulp and every fp32 parity test would fail at 1e-3.)
__device__ __forceinline__ float trunc_tf32(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }

// Converter warps (split form): for a landed fp32 region [begin, end) of a raw stage (16-byte units, any swizzle -- the
// pass is elementwise) write lo = rna_tf32(x - trunc_tf32(x)) to the same offsets of the lo buffer. The raw tile itself is
// the hi operand (see trunc_tf32): it is not rewritten. x - trunc_tf32(x) is exact in fp32 (13 significant bits), so
// hi + lo carries 22 significand bits of x. Four units per thread are loaded before the first is processed.
__device__ __forceinline__ void split_region(const uint8_t* raw, uint8_t* lo, int begin, int end, int ctid, int n_conv) {
  const int stride = n_conv * 16;
  for (int off = begin + ctid * 16; off < end; off += 4 * stride) {
    float4 x[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (off + u * stride < end) x[u] = *reinterpret_cast<const float4*>(raw + off + u * stride);
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (off + u * stride < end) {
        float4 l;
        l.x = rna_tf32(x[u].x - trunc_tf32(x[u].x)); l.y = rna_tf32(x[u].y - trunc_tf32(x[u].y));
        l.z = rna_tf32(x[u].z - trunc_tf32(x[u].z)); l.w = rna_tf32(x[u].w - trunc_tf32(x[u].w));
        *reinterpret_cast<float4*>(lo + off + u * stride) = l;
      }
  }
}

__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// kChunked: some layer of the launch has head_dim > 64 (several K chunks per tile); the common single-chunk case keeps
// its simpler loops (one load iteration per tile).
template <bool kSplit, bool kChunked>
__global__ void __launch_bounds__(kSplit ? kSplitThreads : kThreads, kSplit ? 1 : 2)
accumulate_mma_kernel(const __grid_constant__ MmaParams MP) {
  constexpr int kStageBytesT = kSplit ? kSplitStageBytes : kStageBytes;
  constexpr int kOperandBytes = (kSplit ? kStages + 1 : kStages) * kStageBytesT;     // stages (+ the lo buffer)
  const LaunchParams& P = MP.base;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;                       // 1024-byte alignment for the swizzled tiles
  uint8_t* gen = smem_raw + (base - raw);
  float* sP = reinterpret_cast<float*>(gen + kOperandBytes);
  const uint32_t sP_u32 = base + kOperandBytes;
  const uint32_t bars = sP_u32 + kPBytes;                             // 10 mbarriers + the TMEM base address
  const uint32_t full0 = bars, empty0 = bars + 16, tfull0 = bars + 32, tempty0 = bars + 48;
  const uint32_t lofull = bars + 64, loempty = bars + 72;             // split form: the lo buffer's hand-off
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gen + kOperandBytes + kPBytes + 128);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // The i-th tile of this CTA is first + i * stride.
  int first, count, stride;
  if constexpr (!kChunked) {
    // Equal tiles, interleaved: CTA b takes b, b + G, b + 2G, ... The CTAs of a wave then work on adjacent tiles, i.e.
    // on adjacent 512-byte pieces of the same accumulator token rows (a tile's reduce-add writes 77 of them, 4 * hw
    // bytes apart), so the L2 read-modify-writes of a wave sweep contiguous DRAM ranges instead of landing ~4.7 tiles
    // apart as with contiguous per-CTA ranges (SD-2.1 step 23.1 -> 22.4 us, profiles/r03_ab.json).
    first = blockIdx.x;
    stride = gridDim.x;
    count = (P.total_tiles - first + stride - 1) / stride;
  } else {
    // Tiles of several K-chunk counts: contiguous ranges of equal WEIGHT. (Interleaving measured 5 % slower on SD-1.5's
    // fp32 split form and no faster in fp16, profiles/r03_ab.json.)
    first = tile_at_weight(P, (long long)P.total_weight * blockIdx.x / gridDim.x);
    count = tile_at_weight(P, (long long)P.total_weight * (blockIdx.x + 1) / gridDim.x) - first;
    stride = 1;
  }

  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full0 + 8 * s, 1);
      mbar_init(empty0 + 8 * s, 1);
    }
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull0 + 8 * a, 1);
      mbar_init(tempty0 + 8 * a, 4);       // one arrival per epilogue warp
    }
    mbar_init(lofull, (kSplitThreads - 192) / 32);  // one arrival per converter warp
    mbar_init(loempty, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 5) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // descriptor fetches of the first tile overlap the barrier / TMEM set-up (and, under PDL, the previous kernel's tail)
  if (count > 0 && lane == 0 && (warp == 0 || warp == 4)) {
    int li0 = 0;
    const Tile t0 = decode_tile(P, first, li0);
    if (warp == 0) {
      prefetch_tensormap(&MP.amap[t0.li]);
    } else {
      prefetch_tensormap(&MP.qmap[t0.li]);
      prefetch_tensormap(&MP.kmap[t0.li]);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // Programmatic dependent launch: everything above (barrier init, TMEM allocation) may overlap the tail of the
  // previous kernel on the stream. By default nothing below starts before that kernel has completed and flushed.
  // With `early_loads` (the caller vouches that Q/K were complete before the previous kernel started, DAAM_ACC_EARLY_LOADS)
  // only the accumulator updates wait: loads, MMAs and the first tiles' softmax overlap the previous kernel's tail.
  // Our own dependents may be scheduled as soon as every CTA of this grid is past this point.
  if (!P.early_loads) griddep_wait();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (kSplit && warp >= 6) {
    // ===== converter warps (fp32 projections): landed fp32 tile -> hi (in place) + lo (second buffer) =====
    const int ctid = threadIdx.x - 192, n_conv = kSplitThreads - 192;
    uint8_t* lo = gen + kStages * kStageBytesT;
    int li = 0, j = 0;
    for (int i = 0; i < count; ++i) {
      const Tile t = decode_tile(P, first + i * stride, li);
      const LayerParams& L = P.layer[t.li];
      const int n_chunks = kChunked ? (L.head_dim + 63) >> 6 : 1;
      for (int c = 0; c < n_chunks; ++c, ++j) {
        const int s = j % kStages;
        const int subs = (L.head_dim - 64 * c) > 32 ? 2 : 1;           // live 32-float sub-tiles of this chunk
        mbar_wait(full0 + 8 * s, (uint32_t)(j / kStages) & 1u);         // TMA has landed the raw tiles
        mbar_wait(loempty, ((uint32_t)j & 1u) ^ 1u);                   // the MMAs of the previous chunk have read lo
        uint8_t* stage = gen + s * kStageBytesT;
        split_region(stage, lo, 0, subs * kQBytes, ctid, n_conv);
        split_region(stage, lo, 2 * kQBytes, 2 * kQBytes + subs * kKBytes, ctid, n_conv);
        fence_proxy_async();                           // generic-proxy stores -> visible to the tensor core's reads
        __syncwarp();
        if (lane == 0) mbar_arrive(lofull);
      }
    }
  } else if (warp == 4) {
    // ===== TMA producer =====
    if (lane == 0) {
      int li = 0, j = 0;
      for (int i = 0; i < count; ++i) {
        const Tile t = decode_tile(P, first + i * stride, li);
        const int n_chunks = kChunked ? (P.layer[t.li].head_dim + 63) >> 6 : 1;
        for (int c = 0; c < n_chunks; ++c, ++j) {      // one load iteration = one 64-wide K chunk of one tile
          const int s = j % kStages;
          const uint32_t ph = (uint32_t)(j / kStages) & 1u;
          mbar_wait(empty0 + 8 * s, ph ^ 1u);
          const uint32_t q_dst = base + s * kStageBytesT;
          if constexpr (kSplit) {                      // fp32: up to two 32-float-wide boxes per operand
            const bool two = (P.layer[t.li].head_dim - 64 * c) > 32;    // the second sub-tile has live columns
            const uint32_t k_dst = q_dst + 2 * kQBytes;
            mbar_expect_tx(full0 + 8 * s, two ? kStageBytesT : kStageBytes);
            tma_load_4d(&MP.qmap[t.li], full0 + 8 * s, q_dst, 64 * c, t.head, t.pixel0, t.prompt);
            tma_load_4d(&MP.kmap[t.li], full0 + 8 * s, k_dst, 64 * c, t.head, 0, t.prompt);
            if (two) {
              tma_load_4d(&MP.qmap[t.li], full0 + 8 * s, q_dst + kQBytes, 64 * c + 32, t.head, t.pixel0, t.prompt);
              tma_load_4d(&MP.kmap[t.li], full0 + 8 * s, k_dst + kKBytes, 64 * c + 32, t.head, 0, t.prompt);
            }
          } else {
            const uint32_t k_dst = q_dst + kQBytes;
            mbar_expect_tx(full0 + 8 * s, kStageBytes);
            tma_load_4d(&MP.qmap[t.li], full0 + 8 * s, q_dst, 64 * c, t.head, t.pixel0, t.prompt);
            tma_load_4d(&MP.kmap[t.li], full0 + 8 * s, k_dst, 64 * c, t.head, 0, t.prompt);
          }
        }
      }
    }
  } else if (warp == 5) {
    // ===== MMA issuer =====
    if (lane == 0) {
      int li = 0, j = 0;
      for (int i = 0; i < count; ++i) {
        const Tile t = decode_tile(P, first + i * stride, li);
        const LayerParams& L = P.layer[t.li];
        const int a = i & 1;
        const uint32_t aph = (uint32_t)(i >> 1) & 1u;
        const int n_chunks = kChunked ? (L.head_dim + 63) >> 6 : 1;
        const uint32_t d_tmem = tmem_base + a * kAccCols;
        mbar_wait(tempty0 + 8 * a, aph ^ 1u);          // epilogue has drained this accumulator
        for (int c = 0; c < n_chunks; ++c, ++j) {
          const int s = j % kStages;
          const uint32_t ph = (uint32_t)(j / kStages) & 1u;
          const uint32_t q_src = base + s * kStageBytesT;
          const int cols = min(64, L.head_dim - 64 * c);
          if constexpr (kSplit) {
            mbar_wait(lofull, (uint32_t)j & 1u);       // hi (in place) and lo are written (implies the TMA has landed)
            tc_fence_after();
            // q.k = q_lo.k_hi + q_hi.k_lo + q_hi.k_hi, smallest first; K = 8 floats = 32 bytes per instruction
            const int k_steps = (cols + 7) >> 3;
            const uint32_t q_lo = base + kStages * kStageBytesT, idesc = umma_idesc_tf32();
            const uint32_t qa[3] = {q_lo, q_src, q_src};
            const uint32_t kb[3] = {q_src + 2 * kQBytes, q_lo + 2 * kQBytes, q_src + 2 * kQBytes};
#pragma unroll
            for (int p = 0; p < 3; ++p)
#pragma unroll
              for (int k = 0; k < 8; ++k)
                if (k < k_steps)
                  umma_tf32(d_tmem, umma_desc_sw128(qa[p] + (k >> 2) * kQBytes + 32 * (k & 3)),
                            umma_desc_sw128(kb[p] + (k >> 2) * kKBytes + 32 * (k & 3)), idesc, (c | p | k) != 0);
            umma_commit(loempty);                      // frees the lo buffer ...
          } else {
            mbar_wait(full0 + 8 * s, ph);              // the chunk's operand tiles have landed
            tc_fence_after();
            const int k_steps = (cols + 15) >> 4;      // UMMA_K 16 = 32 bytes along the swizzled row
            const uint32_t k_src = q_src + kQBytes;
            const uint32_t idesc = umma_idesc(L.dtype == DAAM_BF16);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              if (k < k_steps)
                umma_f16(d_tmem, umma_desc_sw128(q_src + 32 * k), umma_desc_sw128(k_src + 32 * k), idesc, (c | k) != 0);
          }
          umma_commit(empty0 + 8 * s);                 // ... and the smem stage once the MMAs have read them
        }
        umma_commit(tfull0 + 8 * a);                   // accumulator ready for the epilogue
      }
    }
  } else if (warp < 4) {
    // ===== epilogue warps: softmax + accumulate =====
    int li = 0;
    const int tid = threadIdx.x;                       // 0..127 == pixel within the tile == TMEM lane
    bool issued = false;
    for (int i = 0; i < count; ++i) {
      const Tile t = decode_tile(P, first + i * stride, li);
      const LayerParams& L = P.layer[t.li];
      const int a = i & 1;
      const uint32_t aph = (uint32_t)(i >> 1) & 1u;
      mbar_wait(tfull0 + 8 * a, aph);
      tc_fence_after();
      float v[kTokensPad];
      const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + a * kAccCols;
#pragma unroll
      for (int c = 0; c < kTokensPad / 16; ++c) tmem_ld16(taddr + c * 16, v + c * 16);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty0 + 8 * a);

      float m = v[0];
#pragma unroll
      for (int j = 1; j < kTokens; ++j) m = fmaxf(m, v[j]);
      const float c = L.scale_log2e, mc = m * c;
      float sum = 0.f;
#pragma unroll
      for (int j = 0; j < kTokens; ++j) {
        v[j] = fast_exp2(fmaf(v[j], c, -mc));
        sum += v[j];
      }
      const float inv = 1.0f / sum;
      // the first accumulator update of this CTA: everything the previous kernel added must be complete and visible
      if (i == 0 && P.early_loads) griddep_wait();

      if (P.rmw_mode == 1) {
        if (tid == 0 && issued) bulk_wait_read0();     // the previous reduce has finished reading sP
        epi_barrier();
#pragma unroll
        for (int j = 0; j < kTokens; ++j) sP[j * kTilePixels + tid] = v[j] * inv;
        fence_proxy_async();                           // generic-proxy writes -> visible to the bulk-async proxy
        epi_barrier();
        if (tid == 0) {
          tma_reduce_add_2d(&MP.amap[t.li], sP_u32, t.pixel0, (t.prompt * L.heads + t.head) * kTokens);
          bulk_commit();
        }
        issued = true;
      } else {
        const int pixel = t.pixel0 + tid;
        if (pixel < L.hw) {
          const long long hw = L.hw;
          float* acc = L.acc + ((long long)(t.prompt * L.heads + t.head) * kTokens) * hw + pixel;
          constexpr int kChunk = 11;
#pragma unroll
          for (int j0 = 0; j0 < kTokens; j0 += kChunk) {
            float old[kChunk];
#pragma unroll
            for (int j = 0; j < kChunk; ++j) old[j] = acc[(j0 + j) * hw];
#pragma unroll
            for (int j = 0; j < kChunk; ++j) acc[(j0 + j) * hw] = fmaf(v[j0 + j], inv, old[j]);
          }
        }
      }
    }
    // shared memory must outlive the reduce's reads; its global writes complete with the grid (same rule as a TMA store)
    if (tid == 0 && issued) bulk_wait_read0();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    __syncwarp();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
  }
}

// ---- host: tensor maps ----------------------------------------------------------------------------------------------
using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                              const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                              CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn get_encode() {
  static EncodeFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  });
  return fn;
}

struct MapKey {
  const void* ptr;
  long long s1, s2, s3;
  int d1, d2, d3, kind;     // kind: 0 q/k 16-bit (dtype in bit 4), 1 accumulator
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && s1 == o.s1 && s2 == o.s2 && s3 == o.s3 && d1 == o.d1 && d2 == o.d2 && d3 == o.d3 &&
           kind == o.kind;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    auto mix = [&h](long long v) { h ^= (size_t)v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2); };
    mix(k.s1); mix(k.s2); mix(k.s3); mix(k.d1); mix(k.d2); mix(k.d3); mix(k.kind);
    return h;
  }
};

// Tensor maps are pure functions of (pointer, shape, strides): cache them, the allocator hands the same Q/K
// addresses back every denoising step.
std::unordered_map<MapKey, CUtensorMap, MapKeyHash>& map_cache() {
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> c;
  return c;
}
std::mutex g_map_mu;

// {head_dim, heads, rows, prompts} view of a projection; box = [box_rows x one 128-byte swizzle span] of one head (64
// 16-bit or 32 fp32 dims), 128B-swizzled; columns beyond head_dim are zero-filled. `promo`: L2 fill granularity.
int make_qk_map(const void* ptr, int dtype, int head_dim, int heads, int rows, int prompts, long long s_head,
                long long s_row, long long s_prompt, int box_rows, CUtensorMapL2promotion promo, CUtensorMap* out) {
  MapKey key{ptr, s_head, s_row, s_prompt, heads, rows, prompts * 1024 + box_rows,
             (dtype << 4) | (head_dim << 8) | ((int)promo << 20)};
  {
    std::lock_guard<std::mutex> lock(g_map_mu);
    auto it = map_cache().find(key);
    if (it != map_cache().end()) { *out = it->second; return DAAM_OK; }
  }
  EncodeFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled is not available from this driver"); return DAAM_E_CUDA; }
  const cuuint64_t es = dtype == DAAM_F32 ? 4 : 2;
  const cuuint64_t dims[4] = {(cuuint64_t)head_dim, (cuuint64_t)heads, (cuuint64_t)rows, (cuuint64_t)prompts};
  auto bytes = [es](long long s) { return (cuuint64_t)(s > 0 ? s : 8) * es; };
  const cuuint64_t strides[3] = {bytes(s_head), bytes(s_row), bytes(s_prompt)};
  const cuuint32_t box[4] = {(cuuint32_t)(128 / es), 1, (cuuint32_t)box_rows, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUtensorMapDataType type = dtype == DAAM_F32    ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                   : dtype == DAAM_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                                        : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  CUresult r = enc(out, type, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(q/k) failed with CUresult %d", (int)r); return DAAM_E_CUDA; }
  std::lock_guard<std::mutex> lock(g_map_mu);
  if (map_cache().size() > 8192) map_cache().clear();
  map_cache()[key] = *out;
  return DAAM_OK;
}

// accumulator as a 2-D fp32 tensor {hw, prompts*heads*77}; box = [77 tokens x 128 pixels], no swizzle.
int make_acc_map(float* acc, int hw, int rows, CUtensorMap* out) {
  MapKey key{acc, 0, 0, 0, hw, rows, 0, 1};
  {
    std::lock_guard<std::mutex> lock(g_map_mu);
    auto it = map_cache().find(key);
    if (it != map_cache().end()) { *out = it->second; return DAAM_OK; }
  }
  EncodeFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled is not available from this driver"); return DAAM_E_CUDA; }
  const cuuint64_t dims[2] = {(cuuint64_t)hw, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)hw * 4};
  const cuuint32_t box[2] = {(cuuint32_t)kTilePixels, (cuuint32_t)kTokens};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, acc, dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(acc) failed with CUresult %d", (int)r); return DAAM_E_CUDA; }
  std::lock_guard<std::mutex> lock(g_map_mu);
  if (map_cache().size() > 8192) map_cache().clear();
  map_cache()[key] = *out;
  return DAAM_OK;
}

std::once_flag g_attr_once[64];                       // the shared-memory attribute is per device

}  // namespace

// Parameter block of one tcgen05 launch, opaque to api.cu (which caches prepared launches by their daam_layer[] input).
struct PreparedMma {
  MmaParams mp;
  int grid, block, smem, variant;                     // variant: bit 0 split (fp32), bit 1 chunked (head_dim > 64)
};
void* prepared_mma_new() { return new PreparedMma; }                 // (aligned new: CUtensorMap is alignas(64))
void prepared_mma_delete(void* p) { delete static_cast<PreparedMma*>(p); }

bool mma_supported(const LayerParams& L) {
  return L.head_dim % 8 == 0 && L.head_dim <= DAAM_MAX_HEAD_DIM && L.vec_ok && L.qs_head > 0 && L.qs_pixel > 0 &&
         L.ks_head > 0 && L.ks_token > 0;
}

// Tensor maps, grid and kernel variant of one pack of layers (all fp32, or all 16-bit). `out`: prepared_mma_new().
int prepare_accumulate_mma(const LaunchParams& p, const DeviceInfo& dev, void* out) {
  if (dev.cc_major != 10) { set_error("the tcgen05 kernel needs an sm_100 device (found sm_%d%d)", dev.cc_major, dev.cc_minor); return DAAM_E_UNSUPPORTED; }
  PreparedMma& pm = *static_cast<PreparedMma*>(out);
  MmaParams& mp = pm.mp;
  mp.base = p;
  const bool split = p.n_layers > 0 && p.layer[0].dtype == DAAM_F32;     // a pack holds one operand class (api.cu)
  bool chunked = false;
  for (int i = 0; i < p.n_layers; ++i) {
    const LayerParams& L = p.layer[i];
    if ((L.dtype == DAAM_F32) != split) { set_error("mixed fp32 / 16-bit layers in one tcgen05 pack"); return DAAM_E_INVALID; }
    // A Q tile reads 128 B of each pixel row (one head) at a 640 / 1280 / 2560-byte row stride: 256-byte L2 fills also
    // bring in the neighbouring head's 128 B, which the CTA owning the same pixels of that head reads in the same wave
    // of the interleaved schedule (SD-2.1 step 22.4 -> 22.2 us, profiles/r03_ab.json)
    if (int rc = make_qk_map(L.q, L.dtype, L.head_dim, L.heads, L.hw, L.n_prompts, L.qs_head, L.qs_pixel, L.qs_prompt, kTilePixels, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, &mp.qmap[i])) return rc;
    if (int rc = make_qk_map(L.k, L.dtype, L.head_dim, L.heads, kTokens, L.n_prompts, L.ks_head, L.ks_token, L.ks_prompt, kTokensPad, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, &mp.kmap[i])) return rc;
    if (int rc = make_acc_map(L.acc, L.hw, L.n_prompts * L.heads * kTokens, &mp.amap[i])) return rc;
    chunked = chunked || L.head_dim > 64;
  }
  cudaError_t attr_err = cudaSuccess;
  std::call_once(g_attr_once[dev.device & 63], [&] {
    auto set = [&](const void* fn, int bytes) {
      cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
      if (e != cudaSuccess) attr_err = e;
    };
    set((const void*)accumulate_mma_kernel<false, false>, kSmemBytes);
    set((const void*)accumulate_mma_kernel<false, true>, kSmemBytes);
    set((const void*)accumulate_mma_kernel<true, false>, kSplitSmemBytes);
    set((const void*)accumulate_mma_kernel<true, true>, kSplitSmemBytes);
  });
  DAAM_CUDA_TRY(attr_err);
  pm.grid = dev.sm_count * (split ? 1 : 2);
  if (pm.grid > p.total_tiles) pm.grid = p.total_tiles;
  pm.block = split ? kSplitThreads : kThreads;
  pm.smem = split ? kSplitSmemBytes : kSmemBytes;
  pm.variant = (split ? 1 : 0) | (chunked ? 2 : 0);
  return DAAM_OK;
}

int launch_prepared_mma(const void* prepared, cudaStream_t stream) {
  const PreparedMma& pm = *static_cast<const PreparedMma*>(prepared);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(pm.grid);
  cfg.blockDim = dim3(pm.block);
  cfg.dynamicSmemBytes = pm.smem;
  cfg.stream = stream;
  // Programmatic stream serialization also inside a stream capture: the launch becomes a kernel node with a programmatic
  // edge from its predecessor (CUDA >= 12.3).
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pm.mp.base.pdl ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  switch (pm.variant) {
    case 0: DAAM_CUDA_TRY(cudaLaunchKernelEx(&cfg, accumulate_mma_kernel<false, false>, pm.mp)); break;
    case 1: DAAM_CUDA_TRY(cudaLaunchKernelEx(&cfg, accumulate_mma_kernel<true, false>, pm.mp)); break;
    case 2: DAAM_CUDA_TRY(cudaLaunchKernelEx(&cfg, accumulate_mma_kernel<false, true>, pm.mp)); break;
    default: DAAM_CUDA_TRY(cudaLaunchKernelEx(&cfg, accumulate_mma_kernel<true, true>, pm.mp)); break;
  }
  DAAM_CUDA_TRY(cudaGetLastError());
  count_launch();
  return DAAM_OK;
}

}  // namespace daam
