// G = X^T X on the 5th-generation tensor cores: tcgen05.mma kind::tf32 with the 3xTF32 split
// (x = hi + lo, G ~= hi^T hi + hi^T lo + lo^T hi), FP32 accumulation in TMEM.
// Reference: sif_functions.py:58-67 (compute_pc); the Gram is all that sklearn's randomized
// SVD needs of X (SURVEY.md section 7 H1, H4).  Specialised for d = 300.
//
// Data flow per CTA (one per SM, persistent over a contiguous range of K = utterance rows):
//   TMA      : X rows [k0, k0+16) arrive as ten 32-column boxes (cols 300..319 zero-filled by
//              the TMA unit) in the canonical MN-major operand layout for 32-bit types,
//              SWIZZLE_128B with a 32-byte base (CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B <->
//              UMMA LayoutType 1, cute Swizzle<2,5,2>; the only MN-major layout tf32 accepts).
//              X is row-major (N, 300), i.e. "MN-major" for both operands of X^T X, so no
//              transpose is ever needed: A = B = the same shared-memory tile.  5-stage ring.
//   workers  : 4 "split" warps compute lo = x - trunc_tf32(x) into a second buffer (element-wise,
//              so swizzle-agnostic) and drain TMEM at segment ends; 4 "corner" warps compute
//              block C (below).  Keeping the two jobs on separate warps matters: on one set of
//              warps their per-stage work was as long as the MMAs of the stage, so the tensor
//              pipe idled whenever a flush put the workers behind.  The MMA ignores the low 13 mantissa bits of its FP32
//              operands (verified bit-for-bit on B200), so "hi" is the raw TMA tile.
//   MMA      : one elected thread issues tcgen05.mma (M = 128) for the upper-triangular blocks
//                 tile A  rows   0..127 x cols   0..303   (N = 160 + 144)  TMEM cols   0..303
//                 tile B  rows 128..255 x cols 128..303   (N = 176)        TMEM cols 304..479
//              with three products (hi*lo, hi*hi, lo*hi) per 8-row K step: 18 MMAs per stage, issued BY A TILE
//              (hi rows 0..127 x {lo, hi}, hi rows 128..255 x {lo, hi}, lo rows 0..127 x hi, lo rows 128..255 x
//              hi) with .collector::a::fill/use/lastuse, so an A tile is fetched from shared memory once per
//              K step instead of once per MMA.  (Shared-memory
//              bandwidth -- operand fetch + the workers below -- is what bounds this kernel.)
//   block C  : the remaining 44x44 block (rows/cols 256..299) does not fit in the 512 TMEM
//              columns next to A and B (it would need 48 more), so the worker warps compute
//              it on the CUDA cores in exact FP32 from the raw tile, 4x4 register blocks.
//   flush    : the tensor core adds each MMA into the FP32 accumulator with truncation, a bias
//              of ~1e-7 per MMA that grows linearly with the K chain (measured 1e-4 relative
//              over 6.7 k rows); every kSeg = 64 stages (1024 rows) the workers drain
//              TMEM (tcgen05.ld) into the CTA's FP32 partial tile in global memory (L2-resident,
//              column-major so that lane = row gives coalesced lines) with round-to-nearest
//              adds, which bounds the bias at ~2e-5 relative.  The partial is read and written with an
//              L2 evict_last policy and X streams through the TMA with evict_first (otherwise the 190 MB
//              of X between two flushes push the 38 MB of partials out to HBM); warp-chunks entirely
//              below the diagonal are skipped (the reduce kernel never reads them).
//   reduce   : a second kernel sums the per-CTA partials in CTA order (deterministic) and
//              mirrors the upper triangle.
#include <cuda.h>

#include "common.cuh"
#include "peer_comm.cuh"

namespace mmb {

namespace tc {

constexpr int kD = 300;
constexpr int kBK = 16;                         // X rows per pipeline stage
constexpr int kStages = 5;
constexpr int kBoxes = 10;                      // 32-column boxes (320 >= 300)
constexpr int kBoxBytes = kBK * 128;            // one box: kBK rows x 128 B
constexpr int kHiBytes = kBoxes * kBoxBytes;    // 20480
constexpr int kStageBytes = 2 * kHiBytes;       // hi + lo
constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/;
constexpr int kSeg = 64;                        // K blocks (1024 rows) accumulated in TMEM between two flushes
constexpr int kThreads = 320;                   // warp0 TMA, warp1 MMA, warps 2-5 split + TMEM flush, warps 6-9 corner block
constexpr int kColsAB = 480, kColsC = 48;
constexpr int kPartialStride = 128 * kColsAB + kColsC * kColsC;   // floats per CTA: tiles A|B, then block C

__device__ __forceinline__ void tma_load_2d_hint(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar,
                                                 uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], "
      "[%4], %5;"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar), "l"(policy) : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ float ld_hint(const float* p, uint64_t policy) {
  float v;
  asm volatile("ld.global.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(policy) : "memory");
  return v;
}
__device__ __forceinline__ void st_hint(float* p, float v, uint64_t policy) {
  asm volatile("st.global.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(p), "f"(v), "l"(policy) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor, MN-major (cute::UMMA::SmemDescriptor bit layout):
// [0,14) start>>4, [16,30) LBO>>4, [32,46) SBO>>4, [46,48) version = 1, [61,64) layout type
// (1 = SWIZZLE_128B_BASE32B).  Canonical layout in 16-byte units: ((8,n),(4,k)):((1,LBO),(8,SBO))
// -- 32 floats contiguous along MN, 4 K rows of 128 B per swizzle atom, K atoms SBO apart,
// 32-column MN blocks LBO apart.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              uint32_t layout_type = 1) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout_type << 61;
  return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 = 1 at [4,6), a/b format
// TF32 = 2 at [7,10)/[10,13), a/b major MN = 1 at bit 15/16, N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t make_idesc(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// The same MMA with a hint for the A-operand collector buffer (SASS UTCHMMA .A_KEEP / .A_REUSE): consecutive MMAs
// that share their A tile (same descriptor, M and K) read it from shared memory once.
enum : int { kCollectDiscard = 0, kCollectFill = 1, kCollectUse = 2, kCollectLastUse = 3 };
template <int MODE>
__device__ __forceinline__ void umma_tf32_c(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  if constexpr (MODE == kCollectFill) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32.collector::a::fill [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  } else if constexpr (MODE == kCollectUse) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32.collector::a::use [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  } else if constexpr (MODE == kCollectLastUse) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32.collector::a::lastuse [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  } else {
    umma_tf32(tmem_d, adesc, bdesc, idesc, accumulate);
  }
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

struct Params {
  int64_t N;
  int n_cta;
  uint32_t lbo, sbo;  // descriptor strides in bytes
  float* partial;
};

__device__ __forceinline__ uint64_t desc_at(uint64_t base, uint32_t saddr) {
  return base | (uint64_t)((saddr >> 4) & 0x3fff);
}

__global__ void __launch_bounds__(kThreads, 1)
    gram_tc_kernel(const __grid_constant__ CUtensorMap tmap, const Params prm) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(smem + kStages * kStageBytes);
  uint32_t* tmem_slot = (uint32_t*)(bars + 3 * kStages + 2);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_full = smem_u32(bars), bar_ready = bar_full + 8 * kStages,
                 bar_empty = bar_ready + 8 * kStages, bar_done = bar_empty + 8 * kStages,
                 bar_free = bar_done + 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const int64_t kblocks = (prm.N + kBK - 1) / kBK;
  const int64_t per = (kblocks + prm.n_cta - 1) / prm.n_cta;
  const int64_t kb0 = (int64_t)blockIdx.x * per;
  int64_t kb1 = kb0 + per;
  if (kb1 > kblocks) kb1 = kblocks;
  const int64_t nkb = kb1 > kb0 ? kb1 - kb0 : 0;
  const int64_t nseg = (nkb + kSeg - 1) / kSeg;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_ready + 8 * s, 4);
      mbar_init(bar_empty + 8 * s, 5);   // MMA commit + the four corner warps (block C reads)
    }
    mbar_init(bar_done, 1);
    mbar_init(bar_free, 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      const uint64_t pol_stream = l2_policy_evict_first();   // X is read once
      for (int64_t i = 0; i < nkb; ++i) {
        const int s = (int)(i % kStages);
        const uint32_t ph = (uint32_t)((i / kStages) & 1);
        mbar_wait(bar_empty + 8 * s, ph ^ 1);
        mbar_expect_tx(bar_full + 8 * s, (uint32_t)kHiBytes);
        const uint32_t dst = smem_base + s * kStageBytes;
        const int row = (int)((kb0 + i) * kBK);
        for (int b = 0; b < kBoxes; ++b)
          tma_load_2d_hint(dst + b * kBoxBytes, &tmap, b * 32, row, bar_full + 8 * s, pol_stream);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      constexpr uint32_t idesc160 = make_idesc(128, 160), idesc144 = make_idesc(128, 144),
                         idesc176 = make_idesc(128, 176);
      const uint32_t blk = prm.lbo;  // byte distance between 32-column blocks
      const uint64_t dbase = make_desc(0, prm.lbo, prm.sbo);
      int64_t i = 0;
      for (int64_t sg = 0; sg < nseg; ++sg) {
        if (sg > 0) {   // the workers have drained the accumulators of the previous segment
          mbar_wait(bar_free, (uint32_t)((sg - 1) & 1));
          tc_fence_after();
        }
        int64_t iend = i + kSeg;
        if (iend > nkb) iend = nkb;
        bool first = true;
        for (; i < iend; ++i) {
          const int s = (int)(i % kStages);
          const uint32_t ph = (uint32_t)((i / kStages) & 1);
          mbar_wait(bar_ready + 8 * s, ph);
          tc_fence_after();
          const uint32_t hi = smem_base + s * kStageBytes, lo = hi + kHiBytes;
#pragma unroll
          for (int ks = 0; ks < kBK / 8; ++ks) {
            const uint32_t koff = ks * 1024;  // 8 K rows = two 4-row swizzle atoms of 512 B
            // The nine MMAs of a K step ordered by A tile, so that each of the four A tiles (hi / lo x rows
            // 0..127 / 128..255) is fetched from shared memory once instead of 9 times in total: the A
            // collector keeps it across the MMAs that share it.  Tile A's 304 columns go as N = 160 + 144
            // rather than 256 + 48: no 24-clock MMA between the long ones (-2.6 %, same bits).
            const uint32_t z = (first && ks == 0) ? 0u : 1u;
            const uint64_t h0 = desc_at(dbase, hi + koff), h4 = desc_at(dbase, hi + koff + 4 * blk),
                           h5 = desc_at(dbase, hi + koff + 5 * blk);
            const uint64_t l0 = desc_at(dbase, lo + koff), l4 = desc_at(dbase, lo + koff + 4 * blk),
                           l5 = desc_at(dbase, lo + koff + 5 * blk);
            umma_tf32_c<kCollectFill>(tmem + 0, h0, l0, idesc160, z);          // hi[0:128]   x lo[0:160]
            umma_tf32_c<kCollectUse>(tmem + 160, h0, l5, idesc144, z);         //             x lo[160:304]
            umma_tf32_c<kCollectUse>(tmem + 0, h0, h0, idesc160, 1u);          //             x hi[0:160]
            umma_tf32_c<kCollectLastUse>(tmem + 160, h0, h5, idesc144, 1u);    //             x hi[160:304]
            umma_tf32_c<kCollectFill>(tmem + 304, h4, l4, idesc176, z);        // hi[128:256] x lo[128:304]
            umma_tf32_c<kCollectLastUse>(tmem + 304, h4, h4, idesc176, 1u);    //             x hi[128:304]
            umma_tf32_c<kCollectFill>(tmem + 0, l0, h0, idesc160, 1u);         // lo[0:128]   x hi[0:160]
            umma_tf32_c<kCollectLastUse>(tmem + 160, l0, h5, idesc144, 1u);    //             x hi[160:304]
            umma_tf32_c<kCollectDiscard>(tmem + 304, l4, h4, idesc176, 1u);    // lo[128:256] x hi[128:304]
          }
          first = false;
          umma_commit(bar_empty + 8 * s);   // frees the stage when these MMAs have read it
        }
        umma_commit(bar_done);              // this segment's accumulators are complete
      }
    }
  } else if (warp < 6) {
    // ===== split warps: lo = x - trunc_tf32(x) for every stage; TMEM flush at segment ends =====
    const int t = threadIdx.x - 64;  // 0..127
    const int q = warp & 3;          // TMEM lane quadrant this warp may read
    const int row = q * 32 + lane;
    float* part = prm.partial + (size_t)blockIdx.x * kPartialStride;
    float* outT = part + row;   // column-major tiles A|B: element (row, c) at part[c * 128 + row]
    const uint64_t pol_keep = l2_policy_evict_last();   // the partial is re-read at every flush: keep it in L2
    int64_t i = 0;
    for (int64_t sg = 0; sg < nseg; ++sg) {
      int64_t iend = i + kSeg;
      if (iend > nkb) iend = nkb;
      for (; i < iend; ++i) {
        const int s = (int)(i % kStages);
        const uint32_t ph = (uint32_t)((i / kStages) & 1);
        mbar_wait(bar_full + 8 * s, ph);
        const uint8_t* stage = smem + s * kStageBytes;
        const float4* hi = (const float4*)stage;
        float4* lo = (float4*)(stage + kHiBytes);
#pragma unroll
        for (int e = 0; e < kHiBytes / 16 / 128; ++e) {
          const float4 x = hi[t + 128 * e];
          float4 l;
          l.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xffffe000u);
          l.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xffffe000u);
          l.z = x.z - __uint_as_float(__float_as_uint(x.z) & 0xffffe000u);
          l.w = x.w - __uint_as_float(__float_as_uint(x.w) & 0xffffe000u);
          lo[t + 128 * e] = l;
        }
        fence_proxy_async();   // generic-proxy writes -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_ready + 8 * s);
      }
      // flush this segment's TMEM accumulators into the FP32 partial (round-to-nearest adds).
      // The partial is stored column-major (column c of tiles A|B = 128 consecutive floats), so
      // with lane = TMEM lane = tile row every global access of the read-modify-write is one
      // fully coalesced 128-byte line per warp (a row-major partial costs 32 lines per access).
      mbar_wait(bar_done, (uint32_t)(sg & 1));
      tc_fence_after();
      for (int c = 0; c < kColsAB; c += 32) {
        // warp-chunks entirely below the diagonal are never read by the reduce kernel: tile A (rows 32 q ..,
        // columns c ..) when c + 32 <= 32 q; tile B (rows 128 + 32 q .., columns 128 + c - 304 ..) likewise
        if (c + 32 <= 32 * q || (c >= 320 && c - 304 + 32 <= 32 * q)) continue;
        float* o = outT + (size_t)c * 128;
        float old[32];
        uint32_t r[32];
        if (sg > 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j) old[j] = ld_hint(o + (size_t)j * 128, pol_keep);
        }
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + c, r);
        if (sg == 0) {
#pragma unroll
          for (int j = 0; j < 32; ++j) st_hint(o + (size_t)j * 128, __uint_as_float(r[j]), pol_keep);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) st_hint(o + (size_t)j * 128, old[j] + __uint_as_float(r[j]), pol_keep);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_free);
    }
    if (nseg == 0)
      for (int c = 0; c < kColsAB; ++c) outT[(size_t)c * 128] = 0.f;
  } else {
    // ===== corner warps: block C (rows/cols 256..299, does not fit in TMEM) in exact FP32 from the
    // raw tile; 11 x 11 grid of 4x4 blocks, upper triangle (66 pairs), dealt round-robin =====
    float* part = prm.partial + (size_t)blockIdx.x * kPartialStride;
    // pair index: packed into two full warps + 2 lanes rather than dealt over the four warps -- the cost of a
    // warp-wide LDS.128 here is its 2-3 shared-memory wavefronts whatever the number of active lanes
    const int pidx = (warp - 6) * 32 + lane;
    int ti = 0, tj = 0;
    const bool has_c = pidx < 66;
    if (has_c) {
      int r = pidx;
      while (r >= 11 - ti) { r -= 11 - ti; ++ti; }
      tj = ti + r;
    }
    float cacc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) cacc[a][b] = 0.f;
    const int ca = 4 * ti, cb = 4 * tj;   // column offsets inside [256, 300)
    const uint32_t offa = (8 + (ca >> 5)) * kBoxBytes + (ca & 7) * 4, cha = (ca & 31) >> 3;
    const uint32_t offb = (8 + (cb >> 5)) * kBoxBytes + (cb & 7) * 4, chb = (cb & 31) >> 3;
    for (int64_t i = 0; i < nkb; ++i) {
      const int s = (int)(i % kStages);
      const uint32_t ph = (uint32_t)((i / kStages) & 1);
      mbar_wait(bar_full + 8 * s, ph);
      const uint8_t* stage = smem + s * kStageBytes;
      if (has_c) {
#pragma unroll
        for (int k = 0; k < kBK; ++k) {
          // 32-byte chunk index is XOR-swizzled with (row & 3)  (SWIZZLE_128B_ATOM_32B)
          const float4 a = *(const float4*)(stage + offa + k * 128 + ((cha ^ (k & 3)) << 5));
          const float4 b = *(const float4*)(stage + offb + k * 128 + ((chb ^ (k & 3)) << 5));
          const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
          for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int v = 0; v < 4; ++v) cacc[u][v] = fmaf(av[u], bv[v], cacc[u][v]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_empty + 8 * s);
    }
    if (has_c) {
      float* cpart = part + 128 * kColsAB;   // 48 x 48 block-C region
#pragma unroll
      for (int u = 0; u < 4; ++u)
        *(float4*)(cpart + (ca + u) * kColsC + cb) = make_float4(cacc[u][0], cacc[u][1], cacc[u][2], cacc[u][3]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
  }
}

// G[i][j] = G[j][i] = sum of the per-CTA partials in CTA order (deterministic).
__global__ void __launch_bounds__(256)
    gram_tc_reduce_kernel(const float* __restrict__ partial, int n_cta, float* __restrict__ G) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= kD * kD) return;
  const int j = idx / kD, i = idx % kD;   // consecutive threads walk a column (coalesced reads)
  if (j < i) return;
  const float* p;
  if (i < 128) p = partial + (size_t)j * 128 + i;
  else if (i < 256) p = partial + (size_t)(304 + (j - 128)) * 128 + (i - 128);
  else p = partial + 128 * kColsAB + (size_t)(i - 256) * kColsC + (j - 256);
  // last use of the partials: read them with evict_first so that the lines the flush pinned (evict_last) stop
  // occupying L2 once the Gram is done
  const uint64_t pol = l2_policy_evict_first();
  float s = 0.f;
  for (int c = 0; c < n_cta; ++c) s += ld_hint(p + (size_t)c * kPartialStride, pol);
  G[(size_t)i * kD + j] = s;
  G[(size_t)j * kD + i] = s;
}

// The same second stage fused with the cross-rank exchange (multi-GPU): sum this rank's per-CTA
// partials straight into its NVLink-visible exchange slot, raise the flags, wait for the peers and
// add all ranks' Grams in rank order -- one launch, no library collective, identical bits on
// every rank.  Launched with one thread per matrix element; the whole grid is co-resident
// (352 CTAs x 256 threads), which the flag wait requires.
__global__ void __launch_bounds__(256)
    gram_tc_reduce_allreduce_kernel(const float* __restrict__ partial, int n_cta, float* __restrict__ G,
                                    const PeerComm comm, int* __restrict__ status) {
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const int nthreads = gridDim.x * blockDim.x;      // cooperative launch: the whole grid is co-resident
  float* mine = (float*)comm_slot(comm, comm.rank);
  const uint64_t pol = l2_policy_evict_first();   // last use of the partials (see gram_tc_reduce_kernel)
  for (int idx = tid; idx < kD * kD; idx += nthreads) {
    const int j = idx / kD, i = idx % kD;
    if (j >= i) {
      const float* p;
      if (i < 128) p = partial + (size_t)j * 128 + i;
      else if (i < 256) p = partial + (size_t)(304 + (j - 128)) * 128 + (i - 128);
      else p = partial + 128 * kColsAB + (size_t)(i - 256) * kColsC + (j - 256);
      float s = 0.f;
      for (int c = 0; c < n_cta; ++c) s += ld_hint(p + (size_t)c * kPartialStride, pol);
      mine[(size_t)i * kD + j] = s;
      mine[(size_t)j * kD + i] = s;
    }
  }
  __syncthreads();
  comm_publish(comm);
  if (!comm_wait(comm)) {
    if (threadIdx.x == 0) atomicOr(status, MMB_STATUS_COMM_TIMEOUT);
    return;
  }
  for (int idx = tid; idx < kD * kD; idx += nthreads) {
    float v[kCommMaxRanks];
#pragma unroll
    for (int r = 0; r < kCommMaxRanks; ++r)
      if (r < comm.world) v[r] = *((const volatile float*)comm_slot(comm, r) + idx);
    float s = v[0];
#pragma unroll
    for (int r = 1; r < kCommMaxRanks; ++r)
      if (r < comm.world) s += v[r];
    G[idx] = s;
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

static int plan(int64_t N) {
  const int64_t kblocks = (N + kBK - 1) / kBK;
  const int sms = sm_count();
  return (int)(kblocks < sms ? (kblocks > 0 ? kblocks : 1) : sms);
}

}  // namespace tc

bool gram_tc_supported(int64_t N, int d) {
  if (d != tc::kD || N < 1) return false;
  static thread_local int cached = -1;
  if (cached < 0) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cached = (major == 10 && tc::encode_fn() != nullptr) ? 1 : 0;
  }
  return cached == 1;
}

size_t gram_tc_workspace_bytes(int64_t N, int d) {
  (void)d;
  return (size_t)tc::plan(N) * tc::kPartialStride * sizeof(float);
}

static int gram_tc_main(const float* X, int64_t N, int d, void* ws, size_t ws_bytes, cudaStream_t st, int* n_cta_out) {
  using namespace tc;
  MMB_REQUIRE(d == kD, "tcgen05 Gram is specialised for d == 300");
  MMB_REQUIRE(N < ((int64_t)1 << 31) - 64, "N too large for 32-bit TMA coordinates");
  const int n_cta = plan(N);
  MMB_REQUIRE(ws_bytes >= (size_t)n_cta * kPartialStride * sizeof(float), "workspace too small");
  EncodeTiledFn enc = encode_fn();
  if (!enc) {
    set_error("gram_tc: cuTensorMapEncodeTiled is not available");
    return MMB_E_UNSUPPORTED;
  }
  CUtensorMap tmap;
  const cuuint64_t gdim[2] = {(cuuint64_t)kD, (cuuint64_t)N};
  const cuuint64_t gstride[1] = {(cuuint64_t)kD * sizeof(float)};
  const cuuint32_t box[2] = {32, (cuuint32_t)kBK};
  const cuuint32_t estride[2] = {1, 1};
  CUresult r = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)X, gdim, gstride, box, estride,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("gram_tc: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return MMB_E_CUDA;
  }
  static bool attr_set = false;
  if (!attr_set) {
    MMB_CUDA(cudaFuncSetAttribute(gram_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    attr_set = true;
  }
  Params prm;
  prm.N = N;
  prm.n_cta = n_cta;
  prm.lbo = kBoxBytes;  // 32-column blocks are kBK*128 bytes apart
  prm.sbo = 512;        // 4-row K atoms (4 x 128 B) are 512 bytes apart
  prm.partial = (float*)ws;
  gram_tc_kernel<<<n_cta, kThreads, kSmemBytes, st>>>(tmap, prm);
  MMB_LAUNCH_CHECK("gram_tc");
  *n_cta_out = n_cta;
  return MMB_OK;
}

int gram_tc(const float* X, int64_t N, int d, float* G, void* ws, size_t ws_bytes, cudaStream_t st) {
  using namespace tc;
  int n_cta = 0;
  const int rc = gram_tc_main(X, N, d, ws, ws_bytes, st, &n_cta);
  if (rc) return rc;
  gram_tc_reduce_kernel<<<(kD * kD + 255) / 256, 256, 0, st>>>((const float*)ws, n_cta, G);
  MMB_LAUNCH_CHECK("gram_tc_reduce");
  return MMB_OK;
}

// Gram + all-reduce over peer memory in two launches: the tcgen05 kernel, then the partial
// reduction fused with the NVLink exchange.
int gram_tc_allreduce(const float* X, int64_t N, int d, float* G, void* ws, size_t ws_bytes, const PeerComm& comm,
                      int* status, cudaStream_t st) {
  using namespace tc;
  int n_cta = 0;
  const int rc = gram_tc_main(X, N, d, ws, ws_bytes, st, &n_cta);
  if (rc) return rc;
  // cooperative launch on an occupancy-bounded grid: the flag wait needs every CTA resident (peer_comm.cuh)
  const int grid = coop_grid((const void*)gram_tc_reduce_allreduce_kernel, 256, 0, (kD * kD + 255) / 256);
  const float* part = (const float*)ws;
  PeerComm c = comm;
  void* args[] = {(void*)&part, (void*)&n_cta, (void*)&G, (void*)&c, (void*)&status};
  MMB_CUDA(cudaLaunchCooperativeKernel((const void*)gram_tc_reduce_allreduce_kernel, dim3(grid), dim3(256), args, 0, st));
  count_launch("gram_tc_reduce_allreduce");
  return MMB_OK;
}

}  // namespace mmb
