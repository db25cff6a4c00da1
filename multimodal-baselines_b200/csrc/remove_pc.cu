// Projection subtraction (reference: sif_functions.py:69-81 remove_pc):
//   npc == 1: XX = X - (X pc^T) * pc          (line 78)
//   npc  > 1: XX = X - (X pc^T) pc            (line 80; all projections taken from X itself)
// HBM-bound streaming pass: one warp per row, the row lives in registers as float4 (read
// once, written once = 2*d*4 bytes per utterance), the components sit in shared memory.
#include "pc_rows.cuh"

namespace mmb {

constexpr int kRmWarps = 8;
constexpr int kRmMaxPc = 8;  // components kept in shared memory per pass

// One warp per row: x[] (and its copy r[]) holds lane's float4 columns lane, lane + 32, ... (zero past d4).
template <int NCH>
__device__ __forceinline__ void load_row(const float4* X4, int64_t i, int d4, int lane, float4 (&x)[NCH],
                                         float4 (&r)[NCH]) {
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    const int k = lane + 32 * c;
    x[c] = k < d4 ? ld_stream(X4 + (size_t)i * d4 + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    r[c] = x[c];
  }
}

template <int NCH>
__global__ void __launch_bounds__(kRmWarps * 32)
    remove_pc_kernel(const float4* __restrict__ X4, int64_t N, int d4, const float4* __restrict__ pc4,
                     int npc, float4* __restrict__ out4) {
  extern __shared__ float4 spc[];  // npc x d4
  for (int k = threadIdx.x; k < npc * d4; k += blockDim.x) spc[k] = pc4[k];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * kRmWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kRmWarps;
  for (int64_t i = warp0; i < N; i += nwarps) {
    float4 x[NCH], r[NCH];
    load_row<NCH>(X4, i, d4, lane, x, r);
    subtract_pcs<NCH>(x, r, spc, npc, d4, lane);
    store_row<NCH>(out4, i, d4, lane, r);
  }
}

// Several component sets against one read of X: out[j] = X - (X pc_j^T) pc_j for every set j of the group,
// each bit for bit what remove_pc_kernel writes for that set alone (npc_j = 0 copies X).  OutV is the output
// vector type: float4 (float32 rows), or double2 (float64 rows: the float32 result, widened on the store).
constexpr int kRmMultiSets = 8;                     // sets per launch
constexpr size_t kRmMultiSmemBytes = 128 * 1024;    // components per launch: one set of 32 x 1024 floats fits

struct RmSets {
  const float4* pc[kRmMultiSets];
  void* out[kRmMultiSets];
  int npc[kRmMultiSets];
  int off[kRmMultiSets];  // first float4 of set j's components in shared memory
  int n;
};

template <int NCH, typename OutV>
__global__ void __launch_bounds__(kRmWarps * 32)
    remove_pc_multi_kernel(const float4* X4, int64_t N, int d4, const RmSets sets) {
  extern __shared__ float4 spc[];
  // the per-set table goes to shared memory: indexing the parameter arrays with a run-time j would copy them
  // to local memory
  __shared__ OutV* s_out[kRmMultiSets];
  __shared__ int s_npc[kRmMultiSets], s_off[kRmMultiSets];
#pragma unroll
  for (int j = 0; j < kRmMultiSets; ++j) {
    if (j < sets.n) {
      for (int k = threadIdx.x; k < sets.npc[j] * d4; k += blockDim.x) spc[sets.off[j] + k] = sets.pc[j][k];
      if (threadIdx.x == 0) {
        s_out[j] = (OutV*)sets.out[j];
        s_npc[j] = sets.npc[j];
        s_off[j] = sets.off[j];
      }
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * kRmWarps + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * kRmWarps;
  for (int64_t i = warp0; i < N; i += nwarps) {
    float4 x[NCH], r[NCH];
    load_row<NCH>(X4, i, d4, lane, x, r);
    for (int j = 0; j < sets.n; ++j) {
      if (j > 0) {
#pragma unroll
        for (int c = 0; c < NCH; ++c) r[c] = x[c];
      }
      subtract_pcs<NCH>(x, r, spc + s_off[j], s_npc[j], d4, lane);
      store_row<NCH>(s_out[j], i, d4, lane, r);
    }
  }
}

}  // namespace mmb

using namespace mmb;

extern "C" int mmb_remove_pc(const float* X, int64_t N, int d, const float* pc, int npc, float* out,
                             mmb_stream_t stream) {
  MMB_REQUIRE(X && pc && out, "null pointer");
  MMB_REQUIRE(d > 0 && d % 4 == 0 && d <= 1024, "d must be a multiple of 4, <= 1024");
  MMB_REQUIRE(npc > 0 && npc <= 32, "npc must be in [1, 32]");
  MMB_REQUIRE(N >= 0, "negative size");
  if (N == 0) return MMB_OK;
  const int d4 = d / 4, nch = (d4 + 31) / 32;
  int64_t blocks = ceil_div(N, kRmWarps);
  int64_t cap = (int64_t)sm_count() * 8;
  const int grid = (int)(blocks < cap ? blocks : cap);
  const size_t smem = (size_t)npc * d4 * sizeof(float4);
  cudaStream_t st = as_stream(stream);
  // more than 48 KB of components (npc * d > 12288, e.g. npc = 32 at d >= 388) needs the opt-in at every NCH
#define RM_LAUNCH(NCH)                                                                                       \
  do {                                                                                                       \
    if (smem > 48 * 1024)                                                                                    \
      MMB_CUDA(cudaFuncSetAttribute(remove_pc_kernel<NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                    (int)smem));                                                             \
    remove_pc_kernel<NCH><<<grid, kRmWarps * 32, smem, st>>>((const float4*)X, N, d4, (const float4*)pc,     \
                                                            npc, (float4*)out);                              \
  } while (0)
  switch (nch) {
    case 1: RM_LAUNCH(1); break;
    case 2: RM_LAUNCH(2); break;
    case 3: RM_LAUNCH(3); break;
    case 4: RM_LAUNCH(4); break;
    default: RM_LAUNCH(8);
  }
#undef RM_LAUNCH
  MMB_LAUNCH_CHECK("remove_pc");
  return MMB_OK;
}

namespace mmb {

// mmb_remove_pc_multi with out[j] float32 (f64 = false) or float64 (f64 = true, the host-buffer sweep's staging).
int remove_pc_multi(const float* X, int64_t N, int d, int P, const float* const* pc, const int* npc,
                    void* const* out, bool f64, cudaStream_t st) {
  // N == 0 touches no row, so X and out[j] may then be NULL (the data pointer of an empty tensor)
  MMB_REQUIRE(pc && npc && out && (X || N == 0), "null pointer");
  MMB_REQUIRE(d > 0 && d % 4 == 0 && d <= 1024, "d must be a multiple of 4, <= 1024");
  MMB_REQUIRE(P > 0, "P must be >= 1");
  MMB_REQUIRE(N >= 0, "negative size");
  for (int j = 0; j < P; ++j) {
    MMB_REQUIRE(npc[j] >= 0 && npc[j] <= 32, "npc must be in [0, 32]");
    MMB_REQUIRE((out[j] || N == 0) && (pc[j] || npc[j] == 0), "null pointer");
    MMB_REQUIRE(P == 1 || N == 0 || out[j] != X, "out may alias X only when P == 1");
  }
  if (N == 0) return MMB_OK;
  const int d4 = d / 4, nch = (d4 + 31) / 32;
  int64_t blocks = ceil_div(N, kRmWarps);
  int64_t cap = (int64_t)sm_count() * 8;
  const int grid = (int)(blocks < cap ? blocks : cap);
  for (int j0 = 0; j0 < P;) {
    // a group: up to kRmMultiSets consecutive sets whose components fit kRmMultiSmemBytes (a single set always does)
    RmSets sets;
    sets.n = 0;
    size_t smem = 0;
    while (j0 + sets.n < P && sets.n < kRmMultiSets) {
      const int j = j0 + sets.n;
      const size_t bytes = (size_t)npc[j] * d4 * sizeof(float4);
      if (sets.n > 0 && smem + bytes > kRmMultiSmemBytes) break;
      sets.pc[sets.n] = (const float4*)pc[j];
      sets.out[sets.n] = out[j];
      sets.npc[sets.n] = npc[j];
      sets.off[sets.n] = (int)(smem / sizeof(float4));
      smem += bytes;
      ++sets.n;
    }
#define RMM_LAUNCH(NCH, OUTV)                                                                                       \
  do {                                                                                                              \
    if (smem > 48 * 1024)                                                                                           \
      MMB_CUDA(cudaFuncSetAttribute(remove_pc_multi_kernel<NCH, OUTV>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                    (int)kRmMultiSmemBytes));                                                       \
    remove_pc_multi_kernel<NCH, OUTV><<<grid, kRmWarps * 32, smem, st>>>((const float4*)X, N, d4, sets);            \
  } while (0)
#define RMM_DISPATCH(OUTV)               \
  switch (nch) {                         \
    case 1: RMM_LAUNCH(1, OUTV); break;  \
    case 2: RMM_LAUNCH(2, OUTV); break;  \
    case 3: RMM_LAUNCH(3, OUTV); break;  \
    case 4: RMM_LAUNCH(4, OUTV); break;  \
    default: RMM_LAUNCH(8, OUTV);        \
  }
    if (f64) {
      RMM_DISPATCH(double2)
    } else {
      RMM_DISPATCH(float4)
    }
#undef RMM_DISPATCH
#undef RMM_LAUNCH
    MMB_LAUNCH_CHECK("remove_pc_multi");
    j0 += sets.n;
  }
  return MMB_OK;
}

}  // namespace mmb

extern "C" int mmb_remove_pc_multi(const float* X, int64_t N, int d, int P, const float* const* pc, const int* npc,
                                   float* const* out, mmb_stream_t stream) {
  return remove_pc_multi(X, N, d, P, pc, npc, (void* const*)out, false, as_stream(stream));
}
