// Row helpers of the projection X - (X pc^T) pc (reference: sif_functions.py:69-81), shared by the projection
// kernels (remove_pc.cu) and the projecting epilogue of the embed kernels (sif_embed.cu), so that a row projected
// as the gather finishes it is bit for bit the row mmb_remove_pc writes.  One warp per row: lane holds float4
// columns lane, lane + 32, ... of the row.
#pragma once

#include "common.cuh"

namespace mmb {

// r -= sum_p dot(x, pc[p]) pc[p] with every dot taken from x (pc: npc x d4, in shared or global memory); r enters
// as x.
template <int NCH>
__device__ __forceinline__ void subtract_pcs(const float4 (&x)[NCH], float4 (&r)[NCH], const float4* spc, int npc,
                                             int d4, int lane) {
  for (int p = 0; p < npc; ++p) {
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int k = lane + 32 * c;
      if (k < d4) {
        const float4 v = spc[p * d4 + k];
        dot = fmaf(x[c].x, v.x, dot);
        dot = fmaf(x[c].y, v.y, dot);
        dot = fmaf(x[c].z, v.z, dot);
        dot = fmaf(x[c].w, v.w, dot);
      }
    }
    dot = warp_sum(dot);
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int k = lane + 32 * c;
      if (k < d4) {
        const float4 v = spc[p * d4 + k];
        r[c].x = fmaf(-dot, v.x, r[c].x);
        r[c].y = fmaf(-dot, v.y, r[c].y);
        r[c].z = fmaf(-dot, v.z, r[c].z);
        r[c].w = fmaf(-dot, v.w, r[c].w);
      }
    }
  }
}

// subtract_pcs with x itself as r, for the embed kernels' epilogue, where a second row array would not fit the
// registers: every dot is first taken from the unchanged x (lane p keeps dot p; npc <= 32; warp_sum's butterfly gives
// every lane the same sum), then x -= dot_p pc[p] for p in order.  The same fmaf sequences as subtract_pcs, so the
// same bits.
template <int NCH>
__device__ __forceinline__ void subtract_pcs_inplace(float4 (&x)[NCH], const float4* pc, int npc, int d4, int lane) {
  float mine = 0.f;
  for (int p = 0; p < npc; ++p) {
    float dot = 0.f;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int k = lane + 32 * c;
      if (k < d4) {
        const float4 v = pc[p * d4 + k];
        dot = fmaf(x[c].x, v.x, dot);
        dot = fmaf(x[c].y, v.y, dot);
        dot = fmaf(x[c].z, v.z, dot);
        dot = fmaf(x[c].w, v.w, dot);
      }
    }
    dot = warp_sum(dot);
    if (lane == p) mine = dot;
  }
  for (int p = 0; p < npc; ++p) {
    const float dot = __shfl_sync(0xffffffffu, mine, p);
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int k = lane + 32 * c;
      if (k < d4) {
        const float4 v = pc[p * d4 + k];
        x[c].x = fmaf(-dot, v.x, x[c].x);
        x[c].y = fmaf(-dot, v.y, x[c].y);
        x[c].z = fmaf(-dot, v.z, x[c].z);
        x[c].w = fmaf(-dot, v.w, x[c].w);
      }
    }
  }
}

template <int NCH>
__device__ __forceinline__ void store_row(float4* out4, int64_t i, int d4, int lane, const float4 (&r)[NCH]) {
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    const int k = lane + 32 * c;
    if (k < d4) st_stream(out4 + (size_t)i * d4 + k, r[c]);
  }
}

// The same row widened to float64 (one cvt per element): float4 k of the row becomes double2 2k and 2k + 1.
template <int NCH>
__device__ __forceinline__ void store_row(double2* out2, int64_t i, int d4, int lane, const float4 (&r)[NCH]) {
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    const int k = lane + 32 * c;
    if (k < d4) {
      double2* p = out2 + ((size_t)i * d4 + k) * 2;
      __stcs(p, make_double2((double)r[c].x, (double)r[c].y));
      __stcs(p + 1, make_double2((double)r[c].z, (double)r[c].w));
    }
  }
}

}  // namespace mmb
