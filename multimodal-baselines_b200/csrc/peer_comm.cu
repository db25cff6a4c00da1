// Exchange-buffer management (CUDA IPC) and the stand-alone peer all-reduce; see peer_comm.cuh.
#include "peer_comm.cuh"

namespace mmb {

int gram_tc_allreduce(const float* X, int64_t N, int d, float* G, void* ws, size_t ws_bytes, const PeerComm& comm,
                      int* status, cudaStream_t st);
bool gram_tc_supported(int64_t N, int d);
int coop_grid(const void* kernel, int threads, size_t smem, int64_t want);

// Grid-stride, cooperative (see comm_wait): copy x into this rank's slot, publish, wait, then
// x[i] = sum over ranks (rank order) of slot_r[i].  V = T or a 16-byte vector of T.
template <typename T>
struct Vec16;
template <> struct Vec16<float> { typedef float4 type; static constexpr int n = 4; };
template <> struct Vec16<double> { typedef double2 type; static constexpr int n = 2; };
__device__ __forceinline__ float4 vadd(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ double2 vadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }

template <typename T>
__global__ void __launch_bounds__(256)
    peer_allreduce_kernel(T* __restrict__ x, int64_t n, const PeerComm comm, int* __restrict__ status) {
  typedef typename Vec16<T>::type V;
  constexpr int VN = Vec16<T>::n;
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const bool vec = ((uintptr_t)x % 16) == 0;
  const int64_t nv = vec ? n / VN : 0;
  T* mine = (T*)comm_slot(comm, comm.rank);
  for (int64_t i = tid; i < nv; i += nthreads) ((V*)mine)[i] = ((const V*)x)[i];
  for (int64_t i = nv * VN + tid; i < n; i += nthreads) mine[i] = x[i];
  __syncthreads();
  comm_publish(comm);
  if (!comm_wait(comm)) {
    if (threadIdx.x == 0) atomicOr(status, MMB_STATUS_COMM_TIMEOUT);
    return;
  }
  for (int64_t i = tid; i < nv; i += nthreads) {
    V v[kCommMaxRanks];
#pragma unroll
    for (int r = 0; r < kCommMaxRanks; ++r)
      if (r < comm.world) v[r] = __ldcv((const V*)comm_slot(comm, r) + i);   // all peers' loads in flight (ld.cv: never a stale cached line)
    V s = v[0];
#pragma unroll
    for (int r = 1; r < kCommMaxRanks; ++r)
      if (r < comm.world) s = vadd(s, v[r]);                                      // rank order
    ((V*)x)[i] = s;
  }
  for (int64_t i = nv * VN + tid; i < n; i += nthreads) {
    T s = (T)0;
    for (int r = 0; r < comm.world; ++r) s += *((const volatile T*)comm_slot(comm, r) + i);
    x[i] = s;
  }
}

__global__ void peer_abort_kernel(const PeerComm comm) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    __threadfence_system();
    for (int p = 0; p < comm.world; ++p) {
      volatile unsigned long long* flag = (volatile unsigned long long*)((char*)comm.buf[p] + kCommFlagsOffset) +
                                          (comm.epoch & 1ull) * kCommMaxRanks + comm.rank;
      *flag = comm.epoch | kCommAbortBit;
    }
    __threadfence_system();
  }
}

// Largest co-resident grid of `kernel` at `threads` per CTA, capped at `want` CTAs.
int coop_grid(const void* kernel, int threads, size_t smem, int64_t want) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess || per_sm < 1)
    per_sm = 1;
  if (per_sm > 4) per_sm = 4;     // the exchange is latency-bound: a few CTAs per SM are plenty
  const int64_t cap = (int64_t)sm_count() * per_sm;
  const int64_t g = want < cap ? want : cap;
  return (int)(g > 0 ? g : 1);
}

static int make_comm(PeerComm* c, int rank, int world, void* const* bufs, uint64_t epoch) {
  MMB_REQUIRE(world >= 1 && world <= kCommMaxRanks && rank >= 0 && rank < world, "need 0 <= rank < world <= 8");
  MMB_REQUIRE(bufs && epoch > 0, "bufs must be given and epoch must be > 0");
  for (int r = 0; r < kCommMaxRanks; ++r) c->buf[r] = r < world ? bufs[r] : nullptr;
  for (int r = 0; r < world; ++r) MMB_REQUIRE(bufs[r], "null exchange buffer");
  c->rank = rank;
  c->world = world;
  c->epoch = epoch;
  return MMB_OK;
}

}  // namespace mmb

using namespace mmb;

extern "C" size_t mmb_comm_bytes(void) { return kCommBytes; }

extern "C" size_t mmb_comm_slot_bytes(void) { return kCommSlotBytes; }

extern "C" int mmb_comm_alloc(void** buf) {
  MMB_REQUIRE(buf, "null pointer");
  MMB_CUDA(cudaMalloc(buf, kCommBytes));
  MMB_CUDA(cudaMemset(*buf, 0, kCommBytes));
  MMB_CUDA(cudaDeviceSynchronize());
  return MMB_OK;
}

extern "C" int mmb_comm_free(void* buf) {
  if (buf) MMB_CUDA(cudaFree(buf));
  return MMB_OK;
}

extern "C" int mmb_comm_export(void* buf, void* handle64) {
  MMB_REQUIRE(buf && handle64, "null pointer");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
  cudaIpcMemHandle_t h;
  MMB_CUDA(cudaIpcGetMemHandle(&h, buf));
  memcpy(handle64, &h, sizeof(h));
  return MMB_OK;
}

extern "C" int mmb_comm_open(const void* handle64, void** peer_buf) {
  MMB_REQUIRE(handle64 && peer_buf, "null pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, sizeof(h));
  MMB_CUDA(cudaIpcOpenMemHandle(peer_buf, h, cudaIpcMemLazyEnablePeerAccess));
  return MMB_OK;
}

extern "C" int mmb_comm_close(void* peer_buf) {
  if (peer_buf) MMB_CUDA(cudaIpcCloseMemHandle(peer_buf));
  return MMB_OK;
}

extern "C" int mmb_allreduce_peer(void* x, int64_t n, int is_f64, int rank, int world, void* const* bufs,
                                  uint64_t epoch, int* status, mmb_stream_t stream) {
  MMB_REQUIRE(x && status && n > 0, "null pointer / empty vector");
  MMB_REQUIRE((size_t)n * (is_f64 ? 8 : 4) <= kCommSlotBytes, "vector larger than the exchange slot (4 MiB)");
  PeerComm c;
  int rc = make_comm(&c, rank, world, bufs, epoch);
  if (rc) return rc;
  const void* fn = is_f64 ? (const void*)peer_allreduce_kernel<double> : (const void*)peer_allreduce_kernel<float>;
  const int grid = coop_grid(fn, 256, 0, ceil_div(n, 256 * (is_f64 ? 2 : 4)));
  void* args[] = {(void*)&x, (void*)&n, (void*)&c, (void*)&status};
  MMB_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(256), args, 0, as_stream(stream)));
  count_launch("peer_allreduce");
  return MMB_OK;
}

extern "C" int mmb_comm_abort(int rank, int world, void* const* bufs, uint64_t epoch, mmb_stream_t stream) {
  PeerComm c;
  int rc = make_comm(&c, rank, world, bufs, epoch);
  if (rc) return rc;
  peer_abort_kernel<<<1, 32, 0, as_stream(stream)>>>(c);
  MMB_LAUNCH_CHECK("peer_abort");
  return MMB_OK;
}

extern "C" int mmb_gram_allreduce_peer(const float* X, int64_t N, int d, float* G, void* ws, size_t ws_bytes,
                                       int mode, int rank, int world, void* const* bufs, uint64_t epoch,
                                       int* status, mmb_stream_t stream) {
  MMB_REQUIRE(G && status && d > 0 && N >= 0, "bad argument");
  MMB_REQUIRE((size_t)d * d * 4 <= kCommSlotBytes, "d x d Gram larger than the exchange slot");
  PeerComm c;
  int rc = make_comm(&c, rank, world, bufs, epoch);
  if (rc) return rc;
  const bool tc = (mode == MMB_GRAM_TF32X3 || (mode == MMB_GRAM_AUTO && N >= 4096)) && N > 0 && gram_tc_supported(N, d);
  if (tc) {
    MMB_REQUIRE(X && ws, "null pointer");
    return gram_tc_allreduce(X, N, d, G, ws, ws_bytes, c, status, as_stream(stream));
  }
  if (N > 0) {
    rc = mmb_gram(X, N, d, G, ws, ws_bytes, mode == MMB_GRAM_AUTO ? MMB_GRAM_FP32 : mode, stream);
    if (rc) return rc;
  } else {
    MMB_CUDA(cudaMemsetAsync(G, 0, (size_t)d * d * sizeof(float), as_stream(stream)));
  }
  return mmb_allreduce_peer(G, (int64_t)d * d, 0, rank, world, bufs, epoch, status, stream);
}
