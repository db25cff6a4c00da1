// Row machinery shared by the SIF gather kernels (sif_embed.cu, sif_embed_multi.cu): packed FP32 accumulators,
// the per-lane chunk predicates, one gathered row's loads / FMAs / store, and the row-offset width switch.
#pragma once

#include "common.cuh"

namespace mmb {

constexpr int kEmbedWarps = 8;  // warps per CTA

// Packed FP32 pairs: Blackwell issues two FP32 FMAs per lane per instruction (fma.rn.f32x2,
// SASS FFMA2), which halves the FMA issue slots of this issue-bound kernel.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ void ffma2(f32x2& acc, f32x2 a, f32x2 b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}

template <int NCH>
struct RowAcc {
  f32x2 a[NCH][2];
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int c = 0; c < NCH; ++c) a[c][0] = a[c][1] = 0ull;   // bit pattern of (0.f, 0.f)
  }
};

// Which of a lane's NCH row chunks (float4 index lane + 32 c) exist, i.e. lie below d4.
//   NCH <= 4 (exact instantiations: d4 in (32 (NCH-1), 32 NCH]): chunks 0..NCH-2 are always whole, only
//     the last one is partial -> one predicate `tail`;
//   NCH == 8 (serves every d4 in 129..256): any chunk may be absent -> a bit per chunk.
// Absent chunks are neither loaded (they would lie beyond the row, for the last rows beyond the table)
// nor accumulated nor stored.
template <int NCH> struct Live { typedef bool type; };
template <> struct Live<8> { typedef unsigned type; };
template <int NCH>
__device__ __forceinline__ typename Live<NCH>::type make_live(int lane, int d4) {
  if constexpr (NCH <= 4) {
    return lane + 32 * (NCH - 1) < d4;
  } else {
    unsigned m = 0;
#pragma unroll
    for (int c = 0; c < NCH; ++c) m |= (lane + 32 * c < d4 ? 1u : 0u) << c;
    return m;
  }
}
template <int NCH>
__device__ __forceinline__ bool chunk_on(typename Live<NCH>::type live, int c) {
  if constexpr (NCH <= 4) return c + 1 < NCH ? true : live;
  else return (live >> c) & 1u;
}

// One gathered row: v[c] = row[lane + 32 c] (coalesced 16-byte loads through the read-only path).
template <int NCH>
__device__ __forceinline__ void load_row(float4 (&v)[NCH], const char* __restrict__ lane_base, size_t off,
                                         typename Live<NCH>::type live) {
  const float4* p = (const float4*)(lane_base + off);
#pragma unroll
  for (int c = 0; c < NCH; ++c)
    if (chunk_on<NCH>(live, c)) v[c] = __ldg(p + 32 * c);
}
template <int NCH>
__device__ __forceinline__ void fma_row(RowAcc<NCH>& acc, const float4 (&v)[NCH], float w,
                                        typename Live<NCH>::type live) {
  const f32x2 ww = pack2(w, w);
#pragma unroll
  for (int c = 0; c < NCH; ++c)
    if (chunk_on<NCH>(live, c)) {
      ffma2(acc.a[c][0], ww, pack2(v[c].x, v[c].y));
      ffma2(acc.a[c][1], ww, pack2(v[c].z, v[c].w));
    }
}

// Byte offset of a table row: 32-bit when the whole table is < 4 GiB (one IMAD per token-lane,
// computed in parallel by the 32 lanes and then shuffled), 64-bit otherwise.
template <bool WIDE> struct RowOff;
template <> struct RowOff<false> { typedef unsigned type; };
template <> struct RowOff<true> { typedef unsigned long long type; };

template <int NCH>
__device__ __forceinline__ void store_row(float4* __restrict__ out, const RowAcc<NCH>& acc, int cnt,
                                          int lane, int d4) {
  const float div = (float)cnt;  // 0 -> inf/NaN row, as NumPy's true_divide
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    int k = lane + 32 * c;
    if ((NCH <= 4 && c + 1 < NCH) || k < d4) {
      float4 r;
      unpack2(acc.a[c][0], r.x, r.y);
      unpack2(acc.a[c][1], r.z, r.w);
      r.x = __fdiv_rn(r.x, div);
      r.y = __fdiv_rn(r.y, div);
      r.z = __fdiv_rn(r.z, div);
      r.w = __fdiv_rn(r.w, div);
      st_stream(out + k, r);
    }
  }
}

}  // namespace mmb
