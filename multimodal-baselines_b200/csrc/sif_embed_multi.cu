// SIF sweep: the weighted average of sif_functions.py:28-56 (weights from seq2weight, lines 8-15) for K
// vocabulary-weight vectors W[0..K-1] over ONE gather of the table rows.
//
// The single-vector embed is bound by the L2 -> SM fabric (every token's d-float row crosses it); a user who sweeps
// the SIF smoothing constant `a` (weights a / (a + p(w))) would pay that K times.  Here every row is read once per
// group of up to KG vectors and FMA'd into KG accumulator sets; what grows with K is KG weight lookups (one sector
// per token, see the workspace layout below), KG FMAs per row element and K outputs.
//
// emb[k] is bit for bit mmb_sif_embed(vocab_w = W[k]) -- the general kernel, not the pre-scaled _ws path:
//   * the same variant rule as launch_embed (sif_embed.cu): few long utterances (L >= 256, N < 16 SMs) take a
//     CTA per utterance with 8 warp partials summed in warp order, everything else a warp per utterance;
//   * rows repeated inside a 32-token chunk are merged with match.any, each group's weight summed per k with the
//     same butterfly warp_sum; singletons keep their own weight;
//   * heads are walked in ascending lane order, one ffma2 per head into each of the KG accumulators;
//   * the divisor is counted per k (count_nonzero of that vector's token weights), stored with __fdiv_rn: a
//     vector with zero entries gets its own count, an all-zero row its own inf/NaN.
// Negative ids wrap like NumPy and get weight 0 for every k; ids outside [-V, V) raise MMB_STATUS_BAD_INDEX.
#include "sif_rows.cuh"

namespace mmb {

// Weight vectors per gather pass by row chunks per lane (NCH = ceil(d / 128)): the accumulators take
// KG * 4 * NCH registers, so KG = 8 for d <= 256, 4 for d <= 512, 2 for d <= 1024.
__host__ __device__ constexpr int multi_group(int nch) { return nch <= 2 ? 8 : (nch <= 4 ? 4 : 2); }
constexpr int kMultiGroupMax = 8;

// Workspace: W (K, V) rewritten per group g (vectors g * Kg .. g * Kg + kw - 1) as a (V, kw) block starting at
// float g * Kg * V, kw = Kg for full groups and the last group's size rounded up to a power of two (padding
// columns 0).  A token's kw weights are then kw * 4 <= 32 contiguous bytes instead of kw sectors of kw lines.
__global__ void __launch_bounds__(256)
    multi_weights_kernel(const float* __restrict__ W, int64_t V, int K, int Kg, int ngroups, int last_w,
                         int64_t total, float* __restrict__ wg) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t block = (int64_t)Kg * V;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += stride) {
    const int g = (int)(e / block);
    const int64_t within = e - g * block;
    const int width = g == ngroups - 1 ? last_w : Kg;
    const int64_t v = within / width;
    const int k = g * Kg + (int)(within - v * width);
    wg[e] = k < K ? __ldg(W + (int64_t)k * V + v) : 0.f;
  }
}

// The KG weights of one token (KG * 4 bytes, aligned to their size).
template <int KG>
__device__ __forceinline__ void load_wk(float (&w)[KG], const float* __restrict__ p) {
  if constexpr (KG >= 4) {
#pragma unroll
    for (int q = 0; q < KG / 4; ++q) {
      const float4 v = __ldg((const float4*)p + q);
      w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
    }
  } else if constexpr (KG == 2) {
    const float2 v = __ldg((const float2*)p);
    w[0] = v.x; w[1] = v.y;
  } else {
    w[0] = __ldg(p);
  }
}

// accumulate_chunk (sif_embed.cu) for KG weight vectors at once: tokens [base, base + 32) of one utterance
// (lane = token), cnt[k] += the number of non-zero weights of vector k among them.
template <int NCH, int KG, int UNROLL, bool WIDE, bool PRE>
__device__ __forceinline__ void accumulate_chunk_multi(RowAcc<NCH> (&acc)[KG], int (&cnt)[KG],
                                                       const char* __restrict__ lane_base, int V, unsigned row_bytes,
                                                       typename Live<NCH>::type tail, const float* __restrict__ wg,
                                                       const int64_t* __restrict__ row_ids, int64_t base, int64_t L,
                                                       int lane, bool& bad, int64_t pre_id) {
  typedef typename RowOff<WIDE>::type off_t;
  const int64_t t = base + lane;
  float w[KG];
#pragma unroll
  for (int k = 0; k < KG; ++k) w[k] = 0.f;
  int row = -1;                       // -1: no token in this lane (past the end / bad index)
  if (t < L) {
    const int64_t id = PRE ? pre_id : __ldcs(row_ids + t);
    const int64_t r = id < 0 ? id + V : id;
    if (r >= 0 && r < V) {
      row = (int)r;
      if (id >= 0) load_wk<KG>(w, wg + (size_t)id * KG);
    } else {
      bad = true;  // NumPy: IndexError
    }
  }
  const off_t off = (off_t)(row < 0 ? 0 : row) * row_bytes;
#pragma unroll
  for (int k = 0; k < KG; ++k) cnt[k] += __popc(__ballot_sync(0xffffffffu, w[k] != 0.f));
  const unsigned grp = __match_any_sync(0xffffffffu, row);
  const bool head = (row >= 0) && (lane == __ffs(grp) - 1);
  const unsigned valid = __ballot_sync(0xffffffffu, row >= 0);
  unsigned heads = __ballot_sync(0xffffffffu, head);
  if (heads != valid) {
    // groups of two or more: their weights summed into the head lane, per vector, in the butterfly order of
    // the single-vector kernel
    unsigned multi = __ballot_sync(0xffffffffu, head && (grp & (grp - 1u)));
    while (multi) {
      const int j = __ffs(multi) - 1;
      multi &= multi - 1u;
      const unsigned gj = __shfl_sync(0xffffffffu, grp, j);
      const bool member = (gj >> lane) & 1u;
#pragma unroll
      for (int k = 0; k < KG; ++k) {
        const float c = warp_sum(member ? w[k] : 0.f);
        if (lane == j) w[k] = c;
      }
    }
  }
  // walk the heads in ascending lane order, UNROLL rows in flight per lane
  while (heads) {
    int j[UNROLL];
    int n = 0;
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      j[u] = heads ? (__ffs(heads) - 1) : 0;
      if (heads) { heads &= heads - 1; ++n; }
    }
    float wj[UNROLL][KG];
    float4 v[UNROLL][NCH];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      if (u < n) {
#pragma unroll
        for (int k = 0; k < KG; ++k) wj[u][k] = __shfl_sync(0xffffffffu, w[k], j[u]);
        const off_t oj = __shfl_sync(0xffffffffu, off, j[u]);
        load_row<NCH>(v[u], lane_base, oj, tail);
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u)
      if (u < n) {
#pragma unroll
        for (int k = 0; k < KG; ++k) fma_row<NCH>(acc[k], v[u], wj[u][k], tail);
      }
  }
}

// Warp per utterance, the next chunk's ids in flight (sif_embed_warp_prefetch_kernel for KG vectors).  emb4 is the
// group's first output; output k of the group is at emb4 + k * N * d4, for k < kn (the rest is padding).
template <int NCH, int KG, int UNROLL, int MINB, bool WIDE>
__global__ void __launch_bounds__(kEmbedWarps * 32, MINB)
    sif_embed_multi_warp_kernel(const float4* __restrict__ table4, int V, int d4, const float* __restrict__ wg,
                                const int64_t* __restrict__ ids, int64_t N, int64_t L, int kn,
                                float4* __restrict__ emb4, int* __restrict__ status) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * kEmbedWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kEmbedWarps;
  const char* lane_base = (const char*)(table4 + lane);
  const unsigned row_bytes = (unsigned)d4 * 16u;
  const typename Live<NCH>::type tail = make_live<NCH>(lane, d4);
  bool bad = false;
  int64_t nid = (warp0 < N && lane < L) ? __ldcs(ids + warp0 * L + lane) : 0;
  for (int64_t i = warp0; i < N; i += nwarps) {
    RowAcc<NCH> acc[KG];
    int cnt[KG];
#pragma unroll
    for (int k = 0; k < KG; ++k) { acc[k].clear(); cnt[k] = 0; }
    const int64_t* row_ids = ids + i * L;
    for (int64_t base = 0; base < L; base += 32) {
      const int64_t id = nid;
      const bool same = base + 32 < L;
      const int64_t ni = same ? i : i + nwarps;
      const int64_t nb = same ? base + 32 : 0;
      nid = (ni < N && nb + lane < L) ? __ldcs(ids + ni * L + nb + lane) : 0;
      accumulate_chunk_multi<NCH, KG, UNROLL, WIDE, true>(acc, cnt, lane_base, V, row_bytes, tail, wg, row_ids, base,
                                                          L, lane, bad, id);
    }
#pragma unroll
    for (int k = 0; k < KG; ++k)
      if (k < kn) store_row<NCH>(emb4 + ((size_t)k * N + i) * d4, acc[k], cnt[k], lane, d4);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(status, MMB_STATUS_BAD_INDEX);
}

// CTA per utterance (few, long utterances): the 8 warps take 32-token chunks round-robin; per output k the warp
// partials go through shared memory and are summed in warp order (sif_embed_cta_kernel, one k at a time so the
// shared footprint is the single-vector kernel's).
template <int NCH, int KG, int UNROLL>
__global__ void __launch_bounds__(kEmbedWarps * 32, 1)
    sif_embed_multi_cta_kernel(const float4* __restrict__ table4, int V, int d4, const float* __restrict__ wg,
                               const int64_t* __restrict__ ids, int64_t N, int64_t L, int kn,
                               float4* __restrict__ emb4, int* __restrict__ status) {
  __shared__ float4 part[kEmbedWarps][NCH * 32];
  __shared__ int part_cnt[kEmbedWarps];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const char* lane_base = (const char*)(table4 + lane);
  const unsigned row_bytes = (unsigned)d4 * 16u;
  const typename Live<NCH>::type tail = make_live<NCH>(lane, d4);
  bool bad = false;
  for (int64_t i = blockIdx.x; i < N; i += gridDim.x) {
    RowAcc<NCH> acc[KG];
    int cnt[KG];
#pragma unroll
    for (int k = 0; k < KG; ++k) { acc[k].clear(); cnt[k] = 0; }
    const int64_t* row_ids = ids + i * L;
    for (int64_t base = 32 * (int64_t)warp; base < L; base += 32 * kEmbedWarps)
      accumulate_chunk_multi<NCH, KG, UNROLL, true, false>(acc, cnt, lane_base, V, row_bytes, tail, wg, row_ids, base,
                                                           L, lane, bad, 0);
#pragma unroll
    for (int k = 0; k < KG; ++k) {
      if (k >= kn) break;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
        if (chunk_on<NCH>(tail, c)) {
          unpack2(acc[k].a[c][0], r.x, r.y);
          unpack2(acc[k].a[c][1], r.z, r.w);
        }
        part[warp][lane + 32 * c] = r;
      }
      if (lane == 0) part_cnt[warp] = cnt[k];
      __syncthreads();
      int total = 0;
#pragma unroll
      for (int w = 0; w < kEmbedWarps; ++w) total += part_cnt[w];
      const float div = (float)total;
      float4* out = emb4 + ((size_t)k * N + i) * d4;
      for (int e = threadIdx.x; e < d4; e += blockDim.x) {
        float4 s = part[0][e];
#pragma unroll
        for (int w = 1; w < kEmbedWarps; ++w) {
          float4 p = part[w][e];
          s.x += p.x; s.y += p.y; s.z += p.z; s.w += p.w;
        }
        s.x = __fdiv_rn(s.x, div); s.y = __fdiv_rn(s.y, div);
        s.z = __fdiv_rn(s.z, div); s.w = __fdiv_rn(s.w, div);
        st_stream(out + e, s);
      }
      __syncthreads();
    }
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(status, MMB_STATUS_BAD_INDEX);
}

// One gather pass: kn (<= KG) vectors whose weights are the (V, KG) block wg, outputs from emb.
template <int NCH, int KG>
static int launch_multi_group(const float* table, int64_t V, int d, const float* wg, const int64_t* ids, int64_t N,
                              int64_t L, int kn, float* emb, int* status, bool few_long, bool wide, int grid,
                              cudaStream_t st, char* kname, size_t kname_len) {
  const int d4 = d / 4;
  // 64 accumulator registers (KG * NCH = 16): one row in flight instead of two (spills otherwise); d > 512 also
  // takes the whole register file (one CTA per SM), as the single-vector kernel's one-row configuration spills.
  // Otherwise as many CTAs per SM as the accumulators allow without spilling: the gather needs warps in flight
  // (B200, 10 M x 64 tokens, d = 300, K = 2: 53.9 ms at 2 CTAs per SM)
  constexpr int UNROLL = (NCH > 4 || KG * NCH >= 16) ? 1 : 2;
  constexpr int MINB = NCH > 4 ? 1 : (KG * NCH <= 2 ? 4 : (KG * NCH <= 6 ? 3 : 2));
  if (few_long) {
    sif_embed_multi_cta_kernel<NCH, KG, UNROLL><<<grid, kEmbedWarps * 32, 0, st>>>(
        (const float4*)table, (int)V, d4, wg, ids, N, L, kn, (float4*)emb, status);
    snprintf(kname, kname_len, "sif_embed_multi_cta_kernel<%d,%d,%d>", NCH, KG, UNROLL);
  } else if (wide) {
    sif_embed_multi_warp_kernel<NCH, KG, UNROLL, MINB, true><<<grid, kEmbedWarps * 32, 0, st>>>(
        (const float4*)table, (int)V, d4, wg, ids, N, L, kn, (float4*)emb, status);
    snprintf(kname, kname_len, "sif_embed_multi_warp_kernel<%d,%d,%d,%d,true>", NCH, KG, UNROLL, MINB);
  } else {
    sif_embed_multi_warp_kernel<NCH, KG, UNROLL, MINB, false><<<grid, kEmbedWarps * 32, 0, st>>>(
        (const float4*)table, (int)V, d4, wg, ids, N, L, kn, (float4*)emb, status);
    snprintf(kname, kname_len, "sif_embed_multi_warp_kernel<%d,%d,%d,%d,false>", NCH, KG, UNROLL, MINB);
  }
  MMB_LAUNCH_CHECK("sif_embed_multi");
  return MMB_OK;
}

template <int NCH>
static int launch_multi(const float* table, int64_t V, int d, const float* vocab_w, int K, const int64_t* ids,
                        int64_t N, int64_t L, float* emb, int* status, float* ws, cudaStream_t st) {
  constexpr int KG = multi_group(NCH);
  const int sms = sm_count();
  const int ngroups = (K + KG - 1) / KG;
  const int last_n = K - (ngroups - 1) * KG;
  int last_w = 1;
  while (last_w < last_n) last_w *= 2;
  const int64_t total = ((int64_t)(ngroups - 1) * KG + last_w) * V;
  const int64_t pblocks = ceil_div(total, 256);
  const int pgrid = (int)(pblocks < (int64_t)sms * 16 ? pblocks : (int64_t)sms * 16);
  multi_weights_kernel<<<pgrid, 256, 0, st>>>(vocab_w, V, K, KG, ngroups, last_w, total, ws);
  MMB_LAUNCH_CHECK("sif_multi_weights");

  // launch_embed's variant rule and grid (sif_embed.cu)
  const bool few_long = (L >= 256) && (N < (int64_t)sms * 16);
  const bool wide = (uint64_t)V * (uint64_t)(d / 4) * 16u >= ((uint64_t)1 << 32);
  const int64_t cap = (int64_t)sms * 8;
  const int64_t blocks = few_long ? N : ceil_div(N, kEmbedWarps);
  const int grid = (int)(blocks < cap ? blocks : cap);
  char kname[96] = "";
  for (int g = 0; g < ngroups; ++g) {
    const int kn = g + 1 < ngroups ? KG : last_n;
    const int kw = g + 1 < ngroups ? KG : last_w;
    const float* wg = ws + (size_t)g * KG * V;
    float* out = emb + (size_t)g * KG * N * d;
    int rc = MMB_OK;
#define MULTI_GROUP(W) \
  rc = launch_multi_group<NCH, W>(table, V, d, wg, ids, N, L, kn, out, status, few_long, wide, grid, st, kname, \
                                  sizeof(kname))
    if (kw == 1) MULTI_GROUP(1);
    else if (kw == 2) MULTI_GROUP(2);
    else if constexpr (KG >= 4) {
      if (kw == 4) MULTI_GROUP(4);
      else if constexpr (KG >= 8) MULTI_GROUP(8);
    }
#undef MULTI_GROUP
    if (rc) return rc;
  }
  note_kernel(1, kname);
  return MMB_OK;
}

}  // namespace mmb

using namespace mmb;

extern "C" size_t mmb_sif_embed_multi_workspace_bytes(int64_t V, int K) {
  // the padded group blocks never exceed K rounded up to the largest group
  if (V <= 0 || K <= 0) return 0;
  return (size_t)V * (size_t)((K + kMultiGroupMax - 1) / kMultiGroupMax * kMultiGroupMax) * sizeof(float);
}

extern "C" int mmb_sif_embed_multi(const float* table, int64_t V, int d, const float* vocab_w, int K, const int64_t* x,
                                   int64_t N, int64_t L, float* emb, int* status, void* ws, size_t ws_bytes,
                                   mmb_stream_t stream) {
  MMB_REQUIRE(d > 0 && d % 4 == 0 && d <= 1024, "d must be a multiple of 4, <= 1024");
  MMB_REQUIRE(V > 0 && V < (int64_t)1 << 31, "V out of range");
  MMB_REQUIRE(K >= 1, "K must be >= 1");
  MMB_REQUIRE(N >= 0 && L >= 0, "negative size");
  if (N == 0) return MMB_OK;   // empty input: nothing to do (pointers may be null)
  MMB_REQUIRE(table && vocab_w && emb && status && ws && (x || L == 0), "null pointer");
  MMB_REQUIRE(ws_bytes >= mmb_sif_embed_multi_workspace_bytes(V, K), "workspace too small");
  MMB_REQUIRE(((uintptr_t)table % 16 == 0) && ((uintptr_t)emb % 16 == 0) && ((uintptr_t)ws % 32 == 0),
              "table / emb must be 16-byte aligned, ws 32-byte aligned");
  cudaStream_t st = as_stream(stream);
  float* wsf = (float*)ws;
  switch ((d / 4 + 31) / 32) {
    case 1: return launch_multi<1>(table, V, d, vocab_w, K, x, N, L, emb, status, wsf, st);
    case 2: return launch_multi<2>(table, V, d, vocab_w, K, x, N, L, emb, status, wsf, st);
    case 3: return launch_multi<3>(table, V, d, vocab_w, K, x, N, L, emb, status, wsf, st);
    case 4: return launch_multi<4>(table, V, d, vocab_w, K, x, N, L, emb, status, wsf, st);
    default: return launch_multi<8>(table, V, d, vocab_w, K, x, N, L, emb, status, wsf, st);
  }
}
