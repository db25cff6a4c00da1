// SIF weighted average (reference: sif_functions.py:8-15 seq2weight, 28-56
// get_weighted_average; sif.py:78-94 glue).
//
// HBM/L2-bound gather + segmented weighted reduction.  One warp owns one utterance: the
// 32 lanes first load 32 token ids (coalesced int64) and look up their weights, then the
// warp walks the tokens in order; for each token the d-float table row is read as
// coalesced float4 (d = 300 -> 75 float4 -> lanes 0..31, 0..31, 0..10) and FMA'd into
// per-lane FP32 accumulators.  The (N, L) weight matrix of the reference never exists in
// the fused path.  Summation is in token order, so the result is deterministic.
//
// Semantics kept from the reference (SURVEY.md section 8a, row A2):
//   * divisor = count_nonzero(w[i, :]) over the whole padded row (pad id 0 counts when its
//     weight is non-zero, as in the POM fixture);
//   * id 0 is an ordinary row of the table;
//   * negative ids: seq2weight gives them weight 0 (line 12) while NumPy's We[x] indexes
//     from the end of the table, so the row is still read and multiplied by 0 (NaN/inf
//     rows propagate exactly as in NumPy);
//   * ids outside [-V, V) are NumPy's IndexError: the kernel skips them and raises
//     MMB_STATUS_BAD_INDEX, which the Python shim turns into IndexError;
//   * an all-zero-weight row divides by zero -> NaN row.
#include "pc_rows.cuh"
#include "sif_rows.cuh"

namespace mmb {

// Epilogue of the embed kernels: the finished row as it is (kPlain), or minus its projection on npc given
// components (mmb_sif_transform), stored as float32 (kProjF32) or widened to float64 (kProjF64; npc may be 0).
// The components are read from global memory through the read-only path: npc * d * 4 bytes (1.2 KB at npc = 1,
// d = 300) stay in L1 next to the gathered rows, and the gather's L1 share -- a capacity number -- loses no shared
// memory carve-out to them.
enum class Epi { kPlain, kProjF32, kProjF64 };
template <Epi E> struct EpiOut { typedef float4 type; };
template <> struct EpiOut<Epi::kProjF64> { typedef double2 type; };

// CTAs per SM (__launch_bounds__ minimum) of the projecting instantiations: the plain kernel's 4 (64 registers) where
// the epilogue fits that budget without spilling, else the most CTAs per SM at which ptxas -v reports no spill (3:
// 80 registers, 2: 128; DESIGN section 4).  The d > 512 warp kernel keeps its 2.  The CTA kernel's plain form sets no
// minimum and ptxas holds it near 64 registers; its projecting forms ask for 2 CTAs per SM (128 registers), or 1.
constexpr int proj_minb(Epi E, int f32, int f64) { return E == Epi::kPlain ? 4 : E == Epi::kProjF32 ? f32 : f64; }
constexpr int prefetch_minb(Epi E, int nch) {
  return proj_minb(E, nch <= 2 ? 4 : 2, nch <= 1 ? 4 : nch == 2 ? 3 : 2);
}
constexpr int prescaled_minb(Epi E, int nch) { return proj_minb(E, nch <= 3 ? 4 : 3, 4); }
constexpr int wide_minb(Epi E, int nch) {
  return proj_minb(E, nch <= 2 ? 4 : nch == 3 ? 3 : 2, nch <= 1 ? 4 : nch <= 3 ? 3 : 2);
}
constexpr int cta_minb(Epi E, int nch) { return E == Epi::kPlain ? 0 : (nch <= 2 ? 2 : 1); }

// Row i of the output.  Projected: x = acc / cnt exactly as store_row forms it (absent chunks 0, as remove_pc's
// load_row reads them), then remove_pc's own subtract_pcs and store, so the row is bit for bit the embed followed
// by mmb_remove_pc.
template <Epi E, int NCH>
__device__ __forceinline__ void finish_row(typename EpiOut<E>::type* __restrict__ out, int64_t i,
                                           const RowAcc<NCH>& acc, int cnt, int lane, int d4,
                                           const float4* __restrict__ pc4, int npc) {
  if constexpr (E == Epi::kPlain) {
    store_row<NCH>(out + (size_t)i * d4, acc, cnt, lane, d4);
  } else {
    const float div = (float)cnt;
    float4 x[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      x[c] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (lane + 32 * c < d4) {
        unpack2(acc.a[c][0], x[c].x, x[c].y);
        unpack2(acc.a[c][1], x[c].z, x[c].w);
        x[c].x = __fdiv_rn(x[c].x, div);
        x[c].y = __fdiv_rn(x[c].y, div);
        x[c].z = __fdiv_rn(x[c].z, div);
        x[c].w = __fdiv_rn(x[c].w, div);
      }
    }
    subtract_pcs_inplace<NCH>(x, pc4, npc, d4, lane);
    store_row<NCH>(out, i, d4, lane, x);
  }
}

// A1: the stand-alone lookup (the reference materialises this matrix; the fused kernel
// below does not).
__global__ void __launch_bounds__(256) seq2weight_kernel(const int64_t* __restrict__ seq,
                                                         const float* __restrict__ mask,
                                                         const float* __restrict__ w4i, int64_t V,
                                                         int64_t n, float* __restrict__ w,
                                                         int* __restrict__ status) {
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  bool bad = false;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    int64_t id = __ldcs(seq + i);
    float m = mask ? __ldcs(mask + i) : 1.f;
    float out = 0.f;
    if (m > 0.f && id >= 0) {
      if (id < V) out = __ldg(w4i + id);
      else bad = true;
    }
    __stcs(w + i, out);
  }
  if (bad) atomicOr(status, MMB_STATUS_BAD_INDEX);
}

// Accumulate tokens [base, base+32) of utterance i (lane = token) into acc; returns the
// number of non-zero weights among them.
//
// Tokens of the chunk that name the same row are merged first (warp match.any):
// sum_j w_j * row == (sum_j w_j) * row, so a row is read once per 32-token chunk however often
// it occurs.  Right-padded batches end in a long run of the pad id (37 % of the tokens of the
// bench workload, 73 % of the POM fixtures), which the reference dutifully gathers and adds one
// by one (pad id 0 is an ordinary row with weight 1.0 in the POM weights), and natural text
// repeats its most frequent words (Zipf: ~18 % of the non-pad tokens of a 32-token chunk).
// The divisor still counts every token's own weight.
// PRE: the lane's id was loaded one chunk ago (`pre_id`, software prefetch by the caller) -- the ids are
// the only operand of this kernel that streams from DRAM, and the weight gather and every row address
// depend on them.
template <int NCH, bool EXPLICIT_W, int UNROLL, bool WIDE, bool PRE = false>
__device__ __forceinline__ int accumulate_chunk(RowAcc<NCH>& acc, const char* __restrict__ lane_base,
                                                int V, unsigned row_bytes, typename Live<NCH>::type tail,
                                                const float* __restrict__ wsrc,
                                                const int64_t* __restrict__ row_ids,
                                                const float* __restrict__ row_w, int64_t base,
                                                int64_t L, int lane, bool& bad, int64_t pre_id = 0) {
  typedef typename RowOff<WIDE>::type off_t;
  const int64_t t = base + lane;
  float w = 0.f;
  int row = -1;                       // -1: no token in this lane (past the end / bad index)
  if (t < L) {
    const int64_t id = PRE ? pre_id : __ldcs(row_ids + t);
    const int64_t r = id < 0 ? id + V : id;
    if (r >= 0 && r < V) {
      row = (int)r;
      w = EXPLICIT_W ? __ldcs(row_w + t) : (id >= 0 ? __ldg(wsrc + id) : 0.f);
    } else {
      bad = true;  // NumPy: IndexError
    }
  }
  const off_t off = (off_t)(row < 0 ? 0 : row) * row_bytes;
  const int cnt = __popc(__ballot_sync(0xffffffffu, w != 0.f));
  // group heads: lowest lane of every set of lanes that hold the same row
  const unsigned grp = __match_any_sync(0xffffffffu, row);
  const bool head = (row >= 0) && (lane == __ffs(grp) - 1);
  const unsigned valid = __ballot_sync(0xffffffffu, row >= 0);
  unsigned heads = __ballot_sync(0xffffffffu, head);
  if (heads == 0xffffffffu) {
    // common case (32 distinct rows): fixed shuffle lanes, no bit scanning
#pragma unroll
    for (int j0 = 0; j0 < 32; j0 += UNROLL) {
      float wj[UNROLL];
      float4 v[UNROLL][NCH];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        wj[u] = __shfl_sync(0xffffffffu, w, j0 + u);
        const off_t oj = __shfl_sync(0xffffffffu, off, j0 + u);
        load_row<NCH>(v[u], lane_base, oj, tail);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) fma_row<NCH>(acc, v[u], wj[u], tail);
    }
    return cnt;
  }
  if (heads != valid) {
    // sum the weights of every group with two or more members into its head lane (fixed
    // butterfly order -> deterministic); singletons keep their own weight
    unsigned multi = __ballot_sync(0xffffffffu, head && (grp & (grp - 1u)));
    while (multi) {
      const int j = __ffs(multi) - 1;
      multi &= multi - 1u;
      const unsigned gj = __shfl_sync(0xffffffffu, grp, j);
      const float c = warp_sum(((gj >> lane) & 1u) ? w : 0.f);
      if (lane == j) w = c;
    }
  }
  // walk the heads, UNROLL rows in flight per lane
  while (heads) {
    int j[UNROLL];
    int n = 0;
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      j[u] = heads ? (__ffs(heads) - 1) : 0;
      if (heads) { heads &= heads - 1; ++n; }
    }
    if (n == UNROLL) {
      float wj[UNROLL];
      float4 v[UNROLL][NCH];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        wj[u] = __shfl_sync(0xffffffffu, w, j[u]);
        const off_t oj = __shfl_sync(0xffffffffu, off, j[u]);
        load_row<NCH>(v[u], lane_base, oj, tail);
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) fma_row<NCH>(acc, v[u], wj[u], tail);
    } else {
      for (int u = 0; u < n; ++u) {
        const float wu = __shfl_sync(0xffffffffu, w, j[u]);
        const off_t oj = __shfl_sync(0xffffffffu, off, j[u]);
        float4 vv[NCH];
        load_row<NCH>(vv, lane_base, oj, tail);
        fma_row<NCH>(acc, vv, wu, tail);
      }
    }
  }
  return cnt;
}

// Warp-per-utterance variant (large N).
// The same kernel with the ids of the NEXT chunk (same utterance, or the warp's next utterance) requested
// before the current chunk's rows are walked.
template <int NCH, int UNROLL, int MINB, Epi E = Epi::kPlain>
__global__ void __launch_bounds__(kEmbedWarps * 32, MINB)
    sif_embed_warp_prefetch_kernel(const float4* __restrict__ table4, int V, int d4, const float* __restrict__ wsrc,
                                   const int64_t* __restrict__ ids, int64_t N, int64_t L,
                                   typename EpiOut<E>::type* __restrict__ emb4, int* __restrict__ status,
                                   const int* __restrict__ only_if_flag = nullptr,
                                   const float4* __restrict__ pc4 = nullptr, int npc = 0) {
  // launched behind sif_embed_prescaled_kernel: work only if that one stood down (flag bit 0 set)
  if (only_if_flag && !(__ldg(only_if_flag) & 1)) return;
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * kEmbedWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kEmbedWarps;
  const char* lane_base = (const char*)(table4 + lane);
  const unsigned row_bytes = (unsigned)d4 * 16u;
  const typename Live<NCH>::type tail = make_live<NCH>(lane, d4);
  bool bad = false;
  int64_t nid = (warp0 < N && lane < L) ? __ldcs(ids + warp0 * L + lane) : 0;
  for (int64_t i = warp0; i < N; i += nwarps) {
    RowAcc<NCH> acc;
    acc.clear();
    int cnt = 0;
    const int64_t* row_ids = ids + i * L;
    for (int64_t base = 0; base < L; base += 32) {
      const int64_t id = nid;
      // next chunk of this warp: the same utterance's next 32 tokens, else the next utterance's first
      const bool same = base + 32 < L;
      const int64_t ni = same ? i : i + nwarps;
      const int64_t nb = same ? base + 32 : 0;
      nid = (ni < N && nb + lane < L) ? __ldcs(ids + ni * L + nb + lane) : 0;
      cnt += accumulate_chunk<NCH, false, UNROLL, false, true>(acc, lane_base, V, row_bytes, tail, wsrc, row_ids,
                                                               nullptr, base, L, lane, bad, id);
    }
    finish_row<E, NCH>(emb4, i, acc, cnt, lane, d4, pc4, npc);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(status, MMB_STATUS_BAD_INDEX);
}

template <int NCH, bool EXPLICIT_W, int UNROLL, int MINB, bool WIDE, Epi E = Epi::kPlain>
__global__ void __launch_bounds__(kEmbedWarps * 32, MINB)
    sif_embed_warp_kernel(const float4* __restrict__ table4, int V, int d4,
                          const float* __restrict__ wsrc, const int64_t* __restrict__ ids,
                          int64_t N, int64_t L, typename EpiOut<E>::type* __restrict__ emb4,
                          int* __restrict__ status, const float4* __restrict__ pc4 = nullptr, int npc = 0) {
  static_assert(E == Epi::kPlain || !EXPLICIT_W, "the projecting epilogue serves the fused-lookup embed only");
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * kEmbedWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kEmbedWarps;
  const char* lane_base = (const char*)(table4 + lane);
  const unsigned row_bytes = (unsigned)d4 * 16u;
  const typename Live<NCH>::type tail = make_live<NCH>(lane, d4);
  bool bad = false;
  for (int64_t i = warp0; i < N; i += nwarps) {
    RowAcc<NCH> acc;
    acc.clear();
    int cnt = 0;
    const int64_t* row_ids = ids + i * L;
    const float* row_w = EXPLICIT_W ? wsrc + i * L : nullptr;
    for (int64_t base = 0; base < L; base += 32)
      cnt += accumulate_chunk<NCH, EXPLICIT_W, UNROLL, WIDE>(acc, lane_base, V, row_bytes, tail, wsrc, row_ids,
                                                             row_w, base, L, lane, bad);
    finish_row<E, NCH>(emb4, i, acc, cnt, lane, d4, pc4, npc);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(status, MMB_STATUS_BAD_INDEX);
}

// ---- large batches: table pre-scaled by the vocabulary weights -------------------------------------------
// For N * L >> V the weights are folded into the table once per call: T'[v] = w[v] * T[v] (one streaming pass
// over the table, 2 * V * d * 4 bytes), after which a token contributes the ROW T'[id] and nothing else:
//   * no weight gather (a random 4-byte read per token = one 32-byte sector through L2 -> L1 and up to 32
//     L1 wavefronts per 32-token chunk),
//   * ONE warp shuffle per gathered row instead of two (row index and multiplicity packed in one word; the
//     shuffles share the L1 data pipe with the row loads -- 20 % of its wavefronts in the general kernel),
//   * a merged group's multiplier is popc(match mask), no reduction loop.
// The divisor needs "weight != 0" per token: the pre-scale pass raises flag bit 0 if ANY vocabulary weight is
// zero (SIF weights a / (a + p) never are); the kernel then returns at once and the general kernel, launched
// behind it, does the work (and returns at once in the usual case) -- no host round trip.  Negative ids keep
// NumPy's semantics: the wrapped row is read and multiplied by 0, and does not count in the divisor.
// Rounding: w * row is rounded once before the sum instead of fused into it -- 2^-24 per term, inside the
// 1e-5 embedding tolerance; the order of the sum is fixed, so the result is deterministic.
constexpr int kRowBits = 26;   // row index below 2^26 (V < 67 M), multiplicity (<= 32) above

__global__ void __launch_bounds__(256)
    prescale_table_kernel(const float4* __restrict__ table4, const float* __restrict__ w, int V, int d4,
                          float4* __restrict__ out4, int* __restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  bool zero = false;
  for (int64_t v = warp0; v < V; v += nwarps) {
    const float wv = __ldg(w + v);
    zero = zero || (wv == 0.f);
    for (int k = lane; k < d4; k += 32) {
      float4 r = ld_stream(table4 + v * d4 + k);
      r.x *= wv; r.y *= wv; r.z *= wv; r.w *= wv;
      out4[v * d4 + k] = r;            // plain store: the rows are about to be gathered (keep them in L2)
    }
  }
  if (zero && lane == 0) atomicOr(flags, 1);
}

template <int NCH, int UNROLL, int MINB, Epi E = Epi::kPlain>
__global__ void __launch_bounds__(kEmbedWarps * 32, MINB)
    sif_embed_prescaled_kernel(const float4* __restrict__ tp4, int V, int d4, const int* __restrict__ flags,
                               const int64_t* __restrict__ ids, int64_t N, int64_t L,
                               typename EpiOut<E>::type* __restrict__ emb4, int* __restrict__ status,
                               const float4* __restrict__ pc4 = nullptr, int npc = 0) {
  if (__ldg(flags) & 1) return;        // a zero vocabulary weight: the general kernel behind this one runs
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * kEmbedWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kEmbedWarps;
  const char* lane_base = (const char*)(tp4 + lane);
  const unsigned row_bytes = (unsigned)d4 * 16u;
  const typename Live<NCH>::type tail = make_live<NCH>(lane, d4);
  bool bad = false;
  int64_t nid = (warp0 < N && lane < L) ? __ldcs(ids + warp0 * L + lane) : 0;
  for (int64_t i = warp0; i < N; i += nwarps) {
    RowAcc<NCH> acc;
    acc.clear();
    int cnt = 0;
    for (int64_t base = 0; base < L; base += 32) {
      const int64_t id = nid;
      const bool same = base + 32 < L;
      const int64_t ni = same ? i : i + nwarps;
      const int64_t nb = same ? base + 32 : 0;
      nid = (ni < N && nb + lane < L) ? __ldcs(ids + ni * L + nb + lane) : 0;      // next chunk's ids in flight
      int row = -1;
      bool counts = false;
      if (base + lane < L) {
        const int64_t r = id < 0 ? id + V : id;
        if (r >= 0 && r < V) {
          row = (int)r;
          counts = id >= 0;            // seq2weight: negative ids get weight 0
        } else {
          bad = true;                  // NumPy: IndexError
        }
      }
      const unsigned nn = __ballot_sync(0xffffffffu, counts);
      cnt += __popc(nn);
      const unsigned grp = __match_any_sync(0xffffffffu, row);
      const bool head = (row >= 0) && (lane == __ffs(grp) - 1);
      const unsigned packed = (unsigned)row | ((unsigned)__popc(grp & nn) << kRowBits);
      unsigned heads = __ballot_sync(0xffffffffu, head);
      while (heads) {
        int j[UNROLL];
        int n = 0;
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
          j[u] = heads ? (__ffs(heads) - 1) : 0;
          if (heads) { heads &= heads - 1; ++n; }
        }
        if (n == UNROLL) {
          float mj[UNROLL];
          float4 v[UNROLL][NCH];
#pragma unroll
          for (int u = 0; u < UNROLL; ++u) {
            const unsigned pj = __shfl_sync(0xffffffffu, packed, j[u]);
            mj[u] = (float)(pj >> kRowBits);
            load_row<NCH>(v[u], lane_base, (pj & ((1u << kRowBits) - 1u)) * row_bytes, tail);
          }
#pragma unroll
          for (int u = 0; u < UNROLL; ++u) fma_row<NCH>(acc, v[u], mj[u], tail);
        } else {
          for (int u = 0; u < n; ++u) {
            const unsigned pj = __shfl_sync(0xffffffffu, packed, j[u]);
            float4 vv[NCH];
            load_row<NCH>(vv, lane_base, (pj & ((1u << kRowBits) - 1u)) * row_bytes, tail);
            fma_row<NCH>(acc, vv, (float)(pj >> kRowBits), tail);
          }
        }
      }
    }
    finish_row<E, NCH>(emb4, i, acc, cnt, lane, d4, pc4, npc);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(status, MMB_STATUS_BAD_INDEX);
}

// Ragged (CSR) variant, SURVEY.md 8f N3: utterance i is tokens[offsets[i] .. offsets[i+1]) -- what is left of a
// right-padded row once its trailing run of the pad id is cut off (utils.py:77-80 pads POM to 1089 / 1357
// tokens: 73 % of that fixture is padding, 37 % of the bench workload).  The reference still sums the pad
// tokens -- the pad id is an ordinary row with an ordinary weight (1.0 in the POM weights) and its weight
// counts in the divisor (sif_functions.py:55) -- so their contribution is added in closed form:
// n_pad * w[pad] * table[pad] to the sum, n_pad to the divisor when w[pad] != 0, n_pad = L_pad - length.
// Result: the padded kernel's, up to the rounding of one multiply instead of per-chunk partial sums.
template <int NCH, int UNROLL, int MINB>
__global__ void __launch_bounds__(kEmbedWarps * 32, MINB)
    sif_embed_ragged_kernel(const float4* __restrict__ table4, int V, int d4, const float* __restrict__ wsrc,
                            const int64_t* __restrict__ tokens, const int64_t* __restrict__ offsets, int64_t N,
                            int64_t L_pad, int64_t pad_id, float4* __restrict__ emb4, int* __restrict__ status) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * kEmbedWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kEmbedWarps;
  const char* lane_base = (const char*)(table4 + lane);
  const unsigned row_bytes = (unsigned)d4 * 16u;
  const typename Live<NCH>::type tail = make_live<NCH>(lane, d4);
  bool bad = false;
  // the pad token: weight by seq2weight's rule (negative id -> 0), row by NumPy's (negative ids wrap)
  const int64_t pad_row = pad_id < 0 ? pad_id + V : pad_id;
  const bool pad_ok = pad_row >= 0 && pad_row < V;
  const float pad_w = (pad_ok && pad_id >= 0) ? __ldg(wsrc + pad_id) : 0.f;
  for (int64_t i = warp0; i < N; i += nwarps) {
    RowAcc<NCH> acc;
    acc.clear();
    int cnt = 0;
    const int64_t o0 = __ldg(offsets + i), o1 = __ldg(offsets + i + 1);
    const int64_t len = o1 - o0;
    for (int64_t base = 0; base < len; base += 32)
      cnt += accumulate_chunk<NCH, false, UNROLL, true>(acc, lane_base, V, row_bytes, tail, wsrc, tokens + o0, nullptr,
                                                        base, len, lane, bad);
    const int64_t n_pad = L_pad - len;
    if (n_pad > 0) {
      if (pad_ok) {
        float4 v[NCH];
        load_row<NCH>(v, lane_base, (size_t)pad_row * row_bytes, tail);
        fma_row<NCH>(acc, v, (float)n_pad * pad_w, tail);
        if (pad_w != 0.f) cnt += (int)n_pad;
      } else {
        bad = true;
      }
    } else if (n_pad < 0) {
      bad = true;    // an utterance longer than the padded length it claims
    }
    store_row<NCH>(emb4 + (size_t)i * d4, acc, cnt, lane, d4);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(status, MMB_STATUS_BAD_INDEX);
}

// padded (N, L) ids -> lengths: index of the last token that is not the pad id, plus one (interior
// occurrences of the pad id -- MOSI's shared OOV row 0 -- stay ordinary tokens).  Warp per row.
__global__ void __launch_bounds__(256)
    ids_lengths_kernel(const int64_t* __restrict__ ids, int64_t N, int64_t L, int64_t pad_id,
                       int64_t* __restrict__ lengths) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = warp0; i < N; i += nwarps) {
    int64_t last = 0;
    for (int64_t base = 0; base < L; base += 32) {
      const int64_t t = base + lane;
      const bool real = t < L && __ldcs(ids + i * L + t) != pad_id;
      const unsigned m = __ballot_sync(0xffffffffu, real);
      if (m) last = base + (32 - __clz(m));
    }
    if (lane == 0) lengths[i] = last;
  }
}

// tokens[offsets[i] + t] = ids[i, t] for t < lengths[i].  Warp per row, coalesced both ways.
__global__ void __launch_bounds__(256)
    ids_compact_kernel(const int64_t* __restrict__ ids, int64_t N, int64_t L, const int64_t* __restrict__ offsets,
                       int64_t* __restrict__ tokens) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = warp0; i < N; i += nwarps) {
    const int64_t o0 = __ldg(offsets + i), len = __ldg(offsets + i + 1) - o0;
    for (int64_t t = lane; t < len; t += 32) tokens[o0 + t] = __ldcs(ids + i * L + t);
  }
}

// offsets[0] = 0, offsets[i + 1] = lengths[0] + ... + lengths[i]: one CTA, chunked scan with a running carry
// (N is at most tens of millions and the conversion runs once per split, next to kernels that take
// milliseconds; 1024 threads x 8 items per round).
__global__ void __launch_bounds__(1024)
    offsets_scan_kernel(const int64_t* __restrict__ lengths, int64_t N, int64_t* __restrict__ offsets) {
  __shared__ long long warp_tot[32];
  __shared__ long long carry_s;
  constexpr int ITEMS = 8;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) { carry_s = 0; offsets[0] = 0; }
  __syncthreads();
  for (int64_t base = 0; base < N; base += 1024 * ITEMS) {
    long long v[ITEMS];
    long long sum = 0;
    const int64_t i0 = base + (int64_t)threadIdx.x * ITEMS;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
      v[k] = (i0 + k < N) ? lengths[i0 + k] : 0;
      sum += v[k];
    }
    long long incl = sum;                       // inclusive scan of the per-thread sums: warp, then CTA
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long n = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += n;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      long long w = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const long long n = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += n;
      }
      warp_tot[lane] = w;                       // inclusive over warps
    }
    __syncthreads();
    long long run = carry_s + (warp ? warp_tot[warp - 1] : 0) + incl - sum;    // exclusive prefix of this thread
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
      run += v[k];
      if (i0 + k < N) offsets[i0 + k + 1] = run;
    }
    __syncthreads();
    if (threadIdx.x == 1023) carry_s = run;
    __syncthreads();
  }
}

// CTA-per-utterance variant (few, long utterances -- the POM shape: 203 x 1357): the 8
// warps take 32-token chunks round-robin and are summed through shared memory in warp
// order, so the result is still deterministic.
// With `offsets` (ragged ids, see sif_embed_ragged_kernel) utterance i is ids[offsets[i] .. offsets[i+1]) followed
// by L - length copies of pad_id, whose closed-form term warp 0 adds.
// Projecting epilogue: the summed row goes back to part[0] and warp 0 reads it in the warp kernels' lane + 32 c
// layout, so that the dot products run in remove_pc's order (the CTA's own thread layout would change it).
template <int NCH, bool EXPLICIT_W, Epi E = Epi::kPlain>
__global__ void __launch_bounds__(kEmbedWarps * 32, cta_minb(E, NCH))
    sif_embed_cta_kernel(const float4* __restrict__ table4, int V, int d4,
                         const float* __restrict__ wsrc, const int64_t* __restrict__ ids, int64_t N,
                         int64_t L, typename EpiOut<E>::type* __restrict__ emb4, int* __restrict__ status,
                         const int64_t* __restrict__ offsets = nullptr, int64_t pad_id = 0,
                         const float4* __restrict__ pc4 = nullptr, int npc = 0) {
  static_assert(E == Epi::kPlain || !EXPLICIT_W, "the projecting epilogue serves the fused-lookup embed only");
  __shared__ float4 part[kEmbedWarps][NCH * 32];
  __shared__ int part_cnt[kEmbedWarps];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const char* lane_base = (const char*)(table4 + lane);
  const unsigned row_bytes = (unsigned)d4 * 16u;
  const typename Live<NCH>::type tail = make_live<NCH>(lane, d4);
  bool bad = false;
  for (int64_t i = blockIdx.x; i < N; i += gridDim.x) {
    RowAcc<NCH> acc;
    acc.clear();
    int cnt = 0;
    const int64_t o0 = offsets ? __ldg(offsets + i) : i * L;
    const int64_t len = offsets ? __ldg(offsets + i + 1) - o0 : L;
    const int64_t* row_ids = ids + o0;
    const float* row_w = EXPLICIT_W ? wsrc + i * L : nullptr;
    for (int64_t base = 32 * (int64_t)warp; base < len; base += 32 * kEmbedWarps)
      cnt += accumulate_chunk<NCH, EXPLICIT_W, 2, true>(acc, lane_base, V, row_bytes, tail, wsrc, row_ids, row_w,
                                                        base, len, lane, bad);
    if (!EXPLICIT_W && offsets && warp == 0) {
      const int64_t n_pad = L - len;
      const int64_t pad_row = pad_id < 0 ? pad_id + V : pad_id;
      if (n_pad > 0 && pad_row >= 0 && pad_row < V) {
        const float pad_w = pad_id >= 0 ? __ldg(wsrc + pad_id) : 0.f;
        float4 v[NCH];
        load_row<NCH>(v, lane_base, (size_t)pad_row * row_bytes, tail);
        fma_row<NCH>(acc, v, (float)n_pad * pad_w, tail);
        if (pad_w != 0.f) cnt += (int)n_pad;
      } else if (n_pad != 0) {
        bad = true;
      }
    }
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
      if (chunk_on<NCH>(tail, c)) {
        unpack2(acc.a[c][0], r.x, r.y);
        unpack2(acc.a[c][1], r.z, r.w);
      }
      part[warp][lane + 32 * c] = r;
    }
    if (lane == 0) part_cnt[warp] = cnt;
    __syncthreads();
    int total = 0;
#pragma unroll
    for (int w = 0; w < kEmbedWarps; ++w) total += part_cnt[w];
    const float div = (float)total;
    for (int k = threadIdx.x; k < d4; k += blockDim.x) {
      float4 s = part[0][k];
#pragma unroll
      for (int w = 1; w < kEmbedWarps; ++w) {
        float4 p = part[w][k];
        s.x += p.x; s.y += p.y; s.z += p.z; s.w += p.w;
      }
      s.x = __fdiv_rn(s.x, div); s.y = __fdiv_rn(s.y, div);
      s.z = __fdiv_rn(s.z, div); s.w = __fdiv_rn(s.w, div);
      if constexpr (E == Epi::kPlain) st_stream(emb4 + (size_t)i * d4 + k, s);
      else part[0][k] = s;           // only this thread reads or writes column k of part[] in this loop
    }
    if constexpr (E != Epi::kPlain) {
      __syncthreads();
      if (warp == 0) {
        float4 x[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c)
          x[c] = lane + 32 * c < d4 ? part[0][lane + 32 * c] : make_float4(0.f, 0.f, 0.f, 0.f);
        subtract_pcs_inplace<NCH>(x, pc4, npc, d4, lane);
        store_row<NCH>(emb4, i, d4, lane, x);
      }
    }
    __syncthreads();
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(status, MMB_STATUS_BAD_INDEX);
}

// " +pc f32" / " +pc f64" after the kernel name of a projecting instantiation (mmb_last_kernel(0))
template <Epi E>
static void note_embed(char (&kname)[96]) {
  if constexpr (E != Epi::kPlain)
    strncat(kname, E == Epi::kProjF32 ? " +pc f32" : " +pc f64", sizeof(kname) - strlen(kname) - 1);
  note_kernel(0, kname);
}

// The variant (CTA per utterance or warp per utterance) is decided on N_total, the batch that N rows are a chunk
// of, so that every chunk of a chunked call runs the kernel the whole batch would.
template <int NCH, bool EXPLICIT_W, Epi E = Epi::kPlain>
static int launch_embed(const float* table, int64_t V, int d, const float* wsrc, const int64_t* ids,
                        int64_t N, int64_t L, void* emb, int* status, cudaStream_t st, int64_t N_total,
                        const float* pc = nullptr, int npc = 0) {
  typedef typename EpiOut<E>::type OutV;
  const int sms = sm_count();
  const int d4 = d / 4;
  const bool few_long = (L >= 256) && (N_total < (int64_t)sms * 16);
  const float4* pc4 = (const float4*)pc;
  char kname[96] = "";
  if (few_long) {
    snprintf(kname, sizeof(kname), "sif_embed_cta_kernel<%d,%s>", NCH, EXPLICIT_W ? "true" : "false");
    int grid = (int)(N < (int64_t)sms * 8 ? N : (int64_t)sms * 8);
    if constexpr (E == Epi::kPlain)
      sif_embed_cta_kernel<NCH, EXPLICIT_W><<<grid, kEmbedWarps * 32, 0, st>>>(
          (const float4*)table, (int)V, d4, wsrc, ids, N, L, (float4*)emb, status);
    else
      sif_embed_cta_kernel<NCH, EXPLICIT_W, E><<<grid, kEmbedWarps * 32, 0, st>>>(
          (const float4*)table, (int)V, d4, wsrc, ids, N, L, (OutV*)emb, status, nullptr, 0, pc4, npc);
  } else {
    // Persistent-style grid: a multiple of the SM count, grid-stride over utterances.
    const int64_t blocks = ceil_div(N, kEmbedWarps);
    const int grid = (int)(blocks < (int64_t)sms * 8 ? blocks : (int64_t)sms * 8);
    // Row pitch = d (dense table).  A 128-byte-aligned pitch (1280 B at d = 300) was measured on
    // B200 and changes nothing (11.88 vs 11.93 ms per 4 M utterances): the L1 wavefront count is
    // not sensitive to where the 512-byte warp reads start.
    const bool wide = (uint64_t)V * (uint64_t)d4 * 16u >= ((uint64_t)1 << 32);
#define EMBED_LAUNCH(U, B, W)                                                                \
  do {                                                                                       \
    sif_embed_warp_kernel<NCH, EXPLICIT_W, U, B, W, E><<<grid, kEmbedWarps * 32, 0, st>>>(   \
        (const float4*)table, (int)V, d4, wsrc, ids, N, L, (OutV*)emb, status, pc4, npc);    \
    snprintf(kname, sizeof(kname), "sif_embed_warp_kernel<%d,%s,%d,%d,%s>", NCH,             \
             EXPLICIT_W ? "true" : "false", U, B, W ? "true" : "false");                     \
  } while (0)
    if constexpr (NCH > 4) {
      // d in 516..1024: 16 accumulator + 32 row registers per row in flight -- one row in flight at
      // 2 CTAs per SM (128 registers) instead of spilling at the d = 300 configuration
      if (wide) EMBED_LAUNCH(1, 2, true);
      else EMBED_LAUNCH(1, 2, false);
    } else if (wide) {
      EMBED_LAUNCH(2, wide_minb(E, NCH), true);
    } else if constexpr (!EXPLICIT_W) {
      // fused lookup: ids of the next chunk prefetched; measured on B200, 4 M utterances: 11.83 ms
      // without the prefetch -> 11.56 ms; also prefetching the next chunk's weight lookups (two chunks
      // ahead) spills at the 64-register budget and takes 16.5 ms -- not kept
      sif_embed_warp_prefetch_kernel<NCH, 2, prefetch_minb(E, NCH), E><<<grid, kEmbedWarps * 32, 0, st>>>(
          (const float4*)table, (int)V, d4, wsrc, ids, N, L, (OutV*)emb, status, nullptr, pc4, npc);
      snprintf(kname, sizeof(kname), "sif_embed_warp_prefetch_kernel<%d,2,%d>", NCH, prefetch_minb(E, NCH));
    } else {
      EMBED_LAUNCH(2, 4, false);
    }
#undef EMBED_LAUNCH
  }
  MMB_LAUNCH_CHECK("sif_embed");
  note_embed<E>(kname);
  return MMB_OK;
}

template <bool EXPLICIT_W, Epi E = Epi::kPlain>
static int dispatch_embed(const float* table, int64_t V, int d, const float* wsrc,
                          const int64_t* ids, int64_t N, int64_t L, void* emb, int* status,
                          cudaStream_t st, int64_t N_total, const float* pc = nullptr, int npc = 0) {
  MMB_REQUIRE(d > 0 && d % 4 == 0 && d <= 1024, "d must be a multiple of 4, <= 1024");
  MMB_REQUIRE(V > 0 && V < (int64_t)1 << 31, "V out of range");
  MMB_REQUIRE(N >= 0 && L >= 0, "negative size");
  if (N == 0) return MMB_OK;   // empty input: nothing to do (pointers may be null)
  MMB_REQUIRE(table && wsrc && emb && status && (ids || L == 0), "null pointer");
  MMB_REQUIRE(((uintptr_t)table % 16 == 0) && ((uintptr_t)emb % 16 == 0), "table/emb must be 16-byte aligned");
  if (N == 0) return MMB_OK;
  const int nch = (d / 4 + 31) / 32;
  switch (nch) {
    case 1: return launch_embed<1, EXPLICIT_W, E>(table, V, d, wsrc, ids, N, L, emb, status, st, N_total, pc, npc);
    case 2: return launch_embed<2, EXPLICIT_W, E>(table, V, d, wsrc, ids, N, L, emb, status, st, N_total, pc, npc);
    case 3: return launch_embed<3, EXPLICIT_W, E>(table, V, d, wsrc, ids, N, L, emb, status, st, N_total, pc, npc);
    case 4: return launch_embed<4, EXPLICIT_W, E>(table, V, d, wsrc, ids, N, L, emb, status, st, N_total, pc, npc);
    default: return launch_embed<8, EXPLICIT_W, E>(table, V, d, wsrc, ids, N, L, emb, status, st, N_total, pc, npc);
  }
}

}  // namespace mmb

using namespace mmb;

extern "C" int mmb_seq2weight(const int64_t* seq, const float* mask, const float* weight4ind,
                              int64_t V, int64_t N, int64_t L, float* w, int* status,
                              mmb_stream_t stream) {
  MMB_REQUIRE(N >= 0 && L >= 0 && V > 0, "bad size");
  const int64_t n = N * L;
  if (n == 0) return MMB_OK;   // empty input: nothing to do (pointers may be null)
  MMB_REQUIRE(seq && weight4ind && w && status, "null pointer");
  int64_t blocks = ceil_div(n, 256 * 4);
  int64_t cap = (int64_t)sm_count() * 16;
  int grid = (int)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
  seq2weight_kernel<<<grid, 256, 0, as_stream(stream)>>>(seq, mask, weight4ind, V, n, w, status);
  MMB_LAUNCH_CHECK("seq2weight");
  return MMB_OK;
}

extern "C" int mmb_weighted_average(const float* table, int64_t V, int d, const int64_t* x,
                                    const float* w, int64_t N, int64_t L, float* emb, int* status,
                                    mmb_stream_t stream) {
  return dispatch_embed<true>(table, V, d, w, x, N, L, emb, status, as_stream(stream), N);
}

extern "C" int mmb_sif_embed(const float* table, int64_t V, int d, const float* vocab_w,
                             const int64_t* x, int64_t N, int64_t L, float* emb, int* status,
                             mmb_stream_t stream) {
  return dispatch_embed<false>(table, V, d, vocab_w, x, N, L, emb, status, as_stream(stream), N);
}

// ---- ragged (CSR) ids, SURVEY.md 8f N3 -----------------------------------------------------------------
extern "C" int mmb_sif_embed_ragged(const float* table, int64_t V, int d, const float* vocab_w,
                                    const int64_t* tokens, const int64_t* offsets, int64_t N, int64_t L_pad,
                                    int64_t pad_id, float* emb, int* status, mmb_stream_t stream) {
  MMB_REQUIRE(d > 0 && d % 4 == 0 && d <= 512, "d must be a multiple of 4, <= 512");
  MMB_REQUIRE(V > 0 && V < (int64_t)1 << 31, "V out of range");
  MMB_REQUIRE(N >= 0 && L_pad >= 0, "negative size");
  if (N == 0) return MMB_OK;
  MMB_REQUIRE(table && vocab_w && offsets && emb && status, "null pointer");
  MMB_REQUIRE(((uintptr_t)table % 16 == 0) && ((uintptr_t)emb % 16 == 0), "table/emb must be 16-byte aligned");
  const int sms = sm_count();
  const int64_t blocks = ceil_div(N, kEmbedWarps);
  const int d4 = d / 4;
  cudaStream_t st = as_stream(stream);
  // few, long utterances (the POM shape): a CTA per utterance, its 8 warps take the 32-token chunks round-robin and
  // are summed in warp order -- parallelism for a handful of rows, and 8 short partial sums instead of one long one
  const bool few_long = (L_pad >= 256) && (N < (int64_t)sms * 16);
  const int grid = few_long ? (int)(N < (int64_t)sms * 8 ? N : (int64_t)sms * 8)
                            : (int)(blocks < (int64_t)sms * 8 ? blocks : (int64_t)sms * 8);
#define RAGGED_LAUNCH(NCH)                                                                                   \
  if (few_long)                                                                                              \
    sif_embed_cta_kernel<NCH, false><<<grid, kEmbedWarps * 32, 0, st>>>(                                     \
        (const float4*)table, (int)V, d4, vocab_w, tokens, N, L_pad, (float4*)emb, status, offsets, pad_id); \
  else                                                                                                       \
    sif_embed_ragged_kernel<NCH, 2, 4><<<grid, kEmbedWarps * 32, 0, st>>>(                                   \
        (const float4*)table, (int)V, d4, vocab_w, tokens, offsets, N, L_pad, pad_id, (float4*)emb, status)
  switch ((d4 + 31) / 32) {
    case 1: RAGGED_LAUNCH(1); break;
    case 2: RAGGED_LAUNCH(2); break;
    case 3: RAGGED_LAUNCH(3); break;
    default: RAGGED_LAUNCH(4); break;
  }
#undef RAGGED_LAUNCH
  MMB_LAUNCH_CHECK("sif_embed_ragged");
  note_kernel(0, few_long ? "sif_embed_cta_kernel (ragged)" : "sif_embed_ragged_kernel");
  return MMB_OK;
}

extern "C" int mmb_ids_lengths(const int64_t* ids, int64_t N, int64_t L, int64_t pad_id, int64_t* lengths,
                               int64_t* offsets, mmb_stream_t stream) {
  MMB_REQUIRE(N >= 0 && L >= 0, "negative size");
  MMB_REQUIRE(offsets && (N == 0 || (lengths && (ids || L == 0))), "null pointer");
  cudaStream_t st = as_stream(stream);
  if (N > 0) {
    const int64_t blocks = ceil_div(N, 8);
    const int grid = (int)(blocks < (int64_t)sm_count() * 8 ? blocks : (int64_t)sm_count() * 8);
    ids_lengths_kernel<<<grid, 256, 0, st>>>(ids, N, L, pad_id, lengths);
    MMB_LAUNCH_CHECK("ids_lengths");
  }
  offsets_scan_kernel<<<1, 1024, 0, st>>>(lengths, N, offsets);
  MMB_LAUNCH_CHECK("offsets_scan");
  return MMB_OK;
}

extern "C" int mmb_ids_compact(const int64_t* ids, int64_t N, int64_t L, const int64_t* offsets, int64_t* tokens,
                               mmb_stream_t stream) {
  MMB_REQUIRE(N >= 0 && L >= 0, "negative size");
  if (N == 0 || L == 0) return MMB_OK;
  MMB_REQUIRE(ids && offsets && tokens, "null pointer");
  const int64_t blocks = ceil_div(N, 8);
  const int grid = (int)(blocks < (int64_t)sm_count() * 8 ? blocks : (int64_t)sm_count() * 8);
  ids_compact_kernel<<<grid, 256, 0, as_stream(stream)>>>(ids, N, L, offsets, tokens);
  MMB_LAUNCH_CHECK("ids_compact");
  return MMB_OK;
}

extern "C" size_t mmb_sif_embed_workspace_bytes(int64_t V, int d, int64_t N, int64_t L) {
  // pre-scaled table + flag word; 0 = the batch is too small for the pre-scale pass to pay (or out of range)
  if (d <= 0 || d % 4 != 0 || d > 512 || V <= 0 || V >= ((int64_t)1 << kRowBits)) return 0;
  if ((uint64_t)V * (uint64_t)d * 4u >= ((uint64_t)1 << 32)) return 0;
  if (L >= 256 && N < (int64_t)sm_count() * 16) return 0;     // few long rows: the CTA-per-utterance kernel
  if (N * L < 8 * V) return 0;
  return (size_t)V * d * sizeof(float) + 256;
}

namespace mmb {
// T' = w * T into ws (+ the zero-weight flag); once per (table, weights), i.e. once per call.
int sif_prescale(const float* table, int64_t V, int d, const float* vocab_w, void* ws, cudaStream_t st) {
  int* flags = (int*)ws;
  float4* tp4 = (float4*)((char*)ws + 256);
  MMB_CUDA(cudaMemsetAsync(flags, 0, sizeof(int), st));
  prescale_table_kernel<<<sm_count() * 8, 256, 0, st>>>((const float4*)table, vocab_w, (int)V, d / 4, tp4, flags);
  MMB_LAUNCH_CHECK("prescale_table");
  return MMB_OK;
}

// The embed pass on a pre-scaled table (ws from sif_prescale) with the general kernel standing by.
template <Epi E = Epi::kPlain>
static int embed_prescaled(const float* table, int64_t V, int d, const float* vocab_w, const void* ws,
                           const int64_t* x, int64_t N, int64_t L, void* emb, int* status, cudaStream_t st,
                           const float* pc = nullptr, int npc = 0) {
  typedef typename EpiOut<E>::type OutV;
  if (N == 0) return MMB_OK;
  const int d4 = d / 4;
  const int* flags = (const int*)ws;
  const float4* tp4 = (const float4*)((const char*)ws + 256);
  const float4* pc4 = (const float4*)pc;
  const int sms = sm_count();
  const int64_t blocks = ceil_div(N, kEmbedWarps);
  const int grid = (int)(blocks < (int64_t)sms * 8 ? blocks : (int64_t)sms * 8);
  char kname[96] = "";
#define PRESCALED_LAUNCH(NCH)                                                                                  \
  do {                                                                                                         \
    sif_embed_prescaled_kernel<NCH, 2, prescaled_minb(E, NCH), E><<<grid, kEmbedWarps * 32, 0, st>>>(          \
        tp4, (int)V, d4, flags, x, N, L, (OutV*)emb, status, pc4, npc);                                        \
    MMB_LAUNCH_CHECK("sif_embed_prescaled");                                                                   \
    sif_embed_warp_prefetch_kernel<NCH, 2, prefetch_minb(E, NCH), E><<<grid, kEmbedWarps * 32, 0, st>>>(       \
        (const float4*)table, (int)V, d4, vocab_w, x, N, L, (OutV*)emb, status, flags, pc4, npc);              \
    MMB_LAUNCH_CHECK("sif_embed_general_standby");                                                             \
    snprintf(kname, sizeof(kname), "sif_embed_prescaled_kernel<%d,2,%d>", NCH, prescaled_minb(E, NCH));       \
  } while (0)
  switch ((d4 + 31) / 32) {
    case 1: PRESCALED_LAUNCH(1); break;
    case 2: PRESCALED_LAUNCH(2); break;
    case 3: PRESCALED_LAUNCH(3); break;
    default: PRESCALED_LAUNCH(4); break;
  }
#undef PRESCALED_LAUNCH
  note_embed<E>(kname);
  return MMB_OK;
}

int sif_embed_prescaled(const float* table, int64_t V, int d, const float* vocab_w, const void* ws, const int64_t* x,
                        int64_t N, int64_t L, float* emb, int* status, cudaStream_t st) {
  return embed_prescaled(table, V, d, vocab_w, ws, x, N, L, emb, status, st);
}

static int check_pc(const float* pc, int npc) {
  MMB_REQUIRE(npc >= 0 && npc <= 32, "npc must be in [0, 32]");
  MMB_REQUIRE(pc || npc == 0, "null pointer");
  MMB_REQUIRE((uintptr_t)pc % 16 == 0, "pc must be 16-byte aligned");
  return MMB_OK;
}

// mmb_sif_transform on N rows of a batch of N_total: the embed with the projection on npc given components (npc x d
// float32 on the device) as its epilogue, out (N, d) float32, or float64 when f64.  scaled: the pre-scaled table of
// sif_prescale for the whole batch, or NULL for the general kernels.
int sif_transform_chunk(const float* table, int64_t V, int d, const float* vocab_w, const void* scaled,
                        const int64_t* x, int64_t N, int64_t L, int64_t N_total, const float* pc, int npc, void* out,
                        bool f64, int* status, cudaStream_t st) {
  if (int rc = check_pc(pc, npc)) return rc;
  if (scaled) {
    if (N == 0) return MMB_OK;
    MMB_REQUIRE(table && vocab_w && x && out && status, "null pointer");
    MMB_REQUIRE(((uintptr_t)table % 16 == 0) && ((uintptr_t)out % 16 == 0) && ((uintptr_t)scaled % 16 == 0),
                "table / out / ws must be 16-byte aligned");
    if (f64) return embed_prescaled<Epi::kProjF64>(table, V, d, vocab_w, scaled, x, N, L, out, status, st, pc, npc);
    if (npc) return embed_prescaled<Epi::kProjF32>(table, V, d, vocab_w, scaled, x, N, L, out, status, st, pc, npc);
    return embed_prescaled(table, V, d, vocab_w, scaled, x, N, L, out, status, st);
  }
  if (f64)
    return dispatch_embed<false, Epi::kProjF64>(table, V, d, vocab_w, x, N, L, out, status, st, N_total, pc, npc);
  if (npc)
    return dispatch_embed<false, Epi::kProjF32>(table, V, d, vocab_w, x, N, L, out, status, st, N_total, pc, npc);
  return dispatch_embed<false>(table, V, d, vocab_w, x, N, L, out, status, st, N_total);
}
}  // namespace mmb

extern "C" int mmb_sif_embed_ws(const float* table, int64_t V, int d, const float* vocab_w, const int64_t* x,
                                int64_t N, int64_t L, float* emb, int* status, void* ws, size_t ws_bytes,
                                mmb_stream_t stream) {
  const size_t need = mmb_sif_embed_workspace_bytes(V, d, N, L);
  if (need == 0 || ws == nullptr || ws_bytes < need || N == 0)
    return mmb_sif_embed(table, V, d, vocab_w, x, N, L, emb, status, stream);
  MMB_REQUIRE(table && vocab_w && x && emb && status, "null pointer");
  MMB_REQUIRE(((uintptr_t)table % 16 == 0) && ((uintptr_t)emb % 16 == 0) && ((uintptr_t)ws % 16 == 0),
              "table / emb / ws must be 16-byte aligned");
  int rc = sif_prescale(table, V, d, vocab_w, ws, as_stream(stream));
  if (rc) return rc;
  return sif_embed_prescaled(table, V, d, vocab_w, ws, x, N, L, emb, status, as_stream(stream));
}

extern "C" int mmb_sif_transform(const float* table, int64_t V, int d, const float* vocab_w, const int64_t* x,
                                 int64_t N, int64_t L, const float* pc, int npc, float* out, int* status, void* ws,
                                 size_t ws_bytes, mmb_stream_t stream) {
  cudaStream_t st = as_stream(stream);
  const size_t need = mmb_sif_embed_workspace_bytes(V, d, N, L);
  const bool scaled = need != 0 && ws != nullptr && ws_bytes >= need && N > 0;
  if (int rc = check_pc(pc, npc)) return rc;
  if (scaled) {
    MMB_REQUIRE(table && vocab_w && (uintptr_t)table % 16 == 0 && (uintptr_t)ws % 16 == 0,
                "table / ws must be non-null and 16-byte aligned");
    const int rc = sif_prescale(table, V, d, vocab_w, ws, st);
    if (rc) return rc;
  }
  return sif_transform_chunk(table, V, d, vocab_w, scaled ? ws : nullptr, x, N, L, N, pc, npc, out, false, status, st);
}
