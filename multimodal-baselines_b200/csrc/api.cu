// libmmb_b200.so: library plumbing (errors, device info, pinned memory), the Gram dispatcher
// and the composed SIF pipelines (device-resident and host-buffer variants).
#include <stdarg.h>
#include <string.h>

#include <vector>

#include "common.cuh"

namespace mmb {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return MMB_E_CUDA;
}

static unsigned long long g_launches = 0;
static char g_last_kernel[8][160];   // last kernel name recorded per stage tag (see note_kernel)

void count_launch(const char*) { __atomic_add_fetch(&g_launches, 1ull, __ATOMIC_RELAXED); }

// Kernels chosen by a run-time dispatch record their (template-expanded) name here so that the
// caller can say WHICH instantiation ran: tag 0 = embed.
void note_kernel(int tag, const char* name) {
  if (tag < 0 || tag >= 8) return;
  strncpy(g_last_kernel[tag], name, sizeof(g_last_kernel[tag]) - 1);
}

int sm_count() {
  static thread_local int cached_dev = -1, cached = 148;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return cached;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) {
      cached = n;
      cached_dev = dev;
    }
  }
  return cached;
}

// implemented in gram_fp32.cu / gram_tc.cu
size_t gram_fp32_workspace_bytes(int64_t N, int d);
int gram_fp32(const float* X, int64_t N, int d, float* G, void* ws, size_t ws_bytes, cudaStream_t st);
size_t gram_tc_workspace_bytes(int64_t N, int d);
int gram_tc(const float* X, int64_t N, int d, float* G, void* ws, size_t ws_bytes, cudaStream_t st);
bool gram_tc_supported(int64_t N, int d);

static int resolve_gram_mode(int64_t N, int d, int mode) {
  // small splits (MOSI / POM sizes) cannot fill a tensor-core pipeline: exact FP32 path
  if (mode == MMB_GRAM_AUTO) return (N >= 4096 && gram_tc_supported(N, d)) ? MMB_GRAM_TF32X3 : MMB_GRAM_FP32;
  return mode;
}

static size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

__global__ void accumulate_kernel(float* __restrict__ acc, const float* __restrict__ x, int n, int first) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) acc[i] = first ? x[i] : acc[i] + x[i];
}

__global__ void f32_to_f64_kernel(const float* __restrict__ in, double* __restrict__ out, int64_t n) {
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = (double)__ldcs(in + i);
}

}  // namespace mmb

using namespace mmb;

extern "C" int mmb_version(void) { return 105; }

extern "C" const char* mmb_last_error(void) { return g_err; }

extern "C" unsigned long long mmb_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

extern "C" const char* mmb_last_kernel(int tag) { return (tag >= 0 && tag < 8) ? g_last_kernel[tag] : ""; }

extern "C" int mmb_device_info(int* sm, int* cc_major, int* cc_minor) {
  int dev = 0;
  MMB_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp p;
  MMB_CUDA(cudaGetDeviceProperties(&p, dev));
  if (sm) *sm = p.multiProcessorCount;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  return MMB_OK;
}

extern "C" int mmb_host_alloc(void** ptr, size_t bytes) {
  MMB_REQUIRE(ptr, "null pointer");
  MMB_CUDA(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
  return MMB_OK;
}

extern "C" int mmb_host_alloc_wc(void** ptr, size_t bytes) {
  MMB_REQUIRE(ptr, "null pointer");
  MMB_CUDA(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocWriteCombined));
  return MMB_OK;
}

extern "C" int mmb_host_free(void* ptr) {
  if (ptr) MMB_CUDA(cudaFreeHost(ptr));
  return MMB_OK;
}

extern "C" size_t mmb_gram_workspace_bytes(int64_t N, int d, int mode) {
  size_t a = gram_fp32_workspace_bytes(N, d);
  if (mode != MMB_GRAM_FP32 && gram_tc_supported(N, d)) {
    size_t b = gram_tc_workspace_bytes(N, d);
    if (b > a) a = b;
  }
  return a;
}

extern "C" int mmb_gram(const float* X, int64_t N, int d, float* G, void* ws, size_t ws_bytes, int mode,
                        mmb_stream_t stream) {
  MMB_REQUIRE(X && G && ws, "null pointer");
  MMB_REQUIRE(d > 0 && d % 4 == 0, "d must be a positive multiple of 4");
  MMB_REQUIRE(N >= 0, "negative N");
  MMB_REQUIRE((uintptr_t)X % 16 == 0, "X must be 16-byte aligned");
  mode = resolve_gram_mode(N, d, mode);
  if (mode == MMB_GRAM_FP32) return gram_fp32(X, N, d, G, ws, ws_bytes, as_stream(stream));
  if (mode == MMB_GRAM_TF32X3) {
    if (!gram_tc_supported(N, d)) {
      set_error("mmb_gram: the tcgen05 path needs d == 300 and N >= 1 on an sm_100 device");
      return MMB_E_UNSUPPORTED;
    }
    return gram_tc(X, N, d, G, ws, ws_bytes, as_stream(stream));
  }
  set_error("mmb_gram: unknown mode %d", mode);
  return MMB_E_INVALID;
}

// ---- composed pipeline, everything resident on the device ---------------------------------
namespace mmb {   // implemented in sif_embed.cu
int sif_prescale(const float* table, int64_t V, int d, const float* vocab_w, void* ws, cudaStream_t st);
int sif_embed_prescaled(const float* table, int64_t V, int d, const float* vocab_w, const void* ws, const int64_t* x,
                        int64_t N, int64_t L, float* emb, int* status, cudaStream_t st);
int sif_transform_chunk(const float* table, int64_t V, int d, const float* vocab_w, const void* scaled,
                        const int64_t* x, int64_t N, int64_t L, int64_t N_total, const float* pc, int npc, void* out,
                        bool f64, int* status, cudaStream_t st);
// implemented in sif_embed_multi.cu / remove_pc.cu (used by mmb_sif_embedding_sweep_host)
int sif_embed_multi_weights(const float* vocab_w, int64_t V, int d, int K, void* ws, cudaStream_t st);
int sif_embed_multi_chunk(const float* table, int64_t V, int d, const void* ws, int K, const int64_t* x,
                          int64_t rows, int64_t L, int64_t N_total, float* emb, int* status, cudaStream_t st);
int remove_pc_multi(const float* X, int64_t N, int d, int P, const float* const* pc, const int* npc,
                    void* const* out, bool f64, cudaStream_t st);
}  // namespace mmb

struct SifWs {
  size_t gram, pc, s0, G, pcv, total;
};
static SifWs sif_ws_layout(int64_t N, int d, int npc) {
  SifWs w;
  const int k = npc + 10;
  size_t off = 0;
  w.gram = off; off += align_up(mmb_gram_workspace_bytes(N, d, MMB_GRAM_AUTO));
  w.pc = off;   off += align_up(mmb_pc_workspace_bytes(d, k));
  w.s0 = off;   off += align_up((size_t)d * k * sizeof(double));
  w.G = off;    off += align_up((size_t)d * d * sizeof(float));
  w.pcv = off;  off += align_up((size_t)(npc > 0 ? npc : 1) * d * sizeof(float));
  w.total = off;
  return w;
}

extern "C" size_t mmb_sif_workspace_bytes(int64_t N, int d, int npc) {
  return sif_ws_layout(N, d, npc > 0 ? npc : 1).total;
}

// Gram -> components -> projection on an (N, d) embedding block already on the device.
static int pc_removal_device(float* emb, int64_t N, int d, int npc, const double* Omega, float* pc_out,
                             float* G_out, void* ws, size_t ws_bytes, int gram_mode, cudaStream_t st) {
  const int k = npc + 10;
  MMB_REQUIRE(k <= 32, "npc must be <= 22");
  SifWs L = sif_ws_layout(N, d, npc);
  MMB_REQUIRE(ws && ws_bytes >= L.total, "workspace too small");
  MMB_REQUIRE(Omega, "Omega (seeded start block) is required when npc > 0");
  char* base = (char*)ws;
  float* G = G_out ? G_out : (float*)(base + L.G);
  float* pc = pc_out ? pc_out : (float*)(base + L.pcv);
  int rc = mmb_gram(emb, N, d, G, base + L.gram, L.pc - L.gram, gram_mode, st);
  if (rc) return rc;
  const double* S0 = Omega;
  const int transposed = N < d;
  if (transposed) {
    rc = mmb_start_block_xt(emb, N, d, Omega, k, (double*)(base + L.s0), st);
    if (rc) return rc;
    S0 = (const double*)(base + L.s0);
  }
  rc = mmb_pc_from_gram(G, d, S0, k, npc, transposed, 7, pc, base + L.pc, L.s0 - L.pc, st);
  if (rc) return rc;
  return mmb_remove_pc(emb, N, d, pc, npc, emb, st);
}

extern "C" int mmb_sif_embedding(const float* table, int64_t V, int d, const float* vocab_w,
                                 const int64_t* x, int64_t N, int64_t L, int npc, const double* Omega,
                                 float* emb, float* pc, float* G, void* ws, size_t ws_bytes,
                                 int gram_mode, int* status, mmb_stream_t stream) {
  // scratch for the pre-scaled table (large batches) sits behind the Gram / solve workspace when the caller
  // provided mmb_sif_workspace_bytes(N, d, npc) + mmb_sif_embed_workspace_bytes(V, d, N, L) bytes
  const size_t base_bytes = align_up(mmb_sif_workspace_bytes(N > 0 ? N : 1, d, npc));
  const size_t scaled_bytes = mmb_sif_embed_workspace_bytes(V, d, N, L);
  int rc;
  if (scaled_bytes && ws && ws_bytes >= base_bytes + scaled_bytes)
    rc = mmb_sif_embed_ws(table, V, d, vocab_w, x, N, L, emb, status, (char*)ws + base_bytes, scaled_bytes, stream);
  else
    rc = mmb_sif_embed(table, V, d, vocab_w, x, N, L, emb, status, stream);
  if (rc || npc <= 0 || N == 0) return rc;
  return pc_removal_device(emb, N, d, npc, Omega, pc, G, ws, ws_bytes, gram_mode, as_stream(stream));
}

// ---- the same call with host buffers --------------------------------------------------------
namespace {
// Staging memory of the *_host entry points comes from a PRIVATE stream-ordered pool per device whose
// release threshold keeps freed blocks for the next call (repeated calls do not pay cudaMalloc again).
// The device's default pool -- and with it every other user of cudaMallocAsync in the process -- is left
// alone; mmb_host_pipeline_trim() hands the cached blocks back to the driver.
cudaMemPool_t g_host_pool[64] = {};

int host_pool(cudaMemPool_t* out) {
  int dev = 0;
  MMB_CUDA(cudaGetDevice(&dev));
  MMB_REQUIRE(dev >= 0 && dev < 64, "device ordinal out of range");
  if (!g_host_pool[dev]) {
    cudaMemPoolProps props = {};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t pool;
    MMB_CUDA(cudaMemPoolCreate(&pool, &props));
    uint64_t keep = UINT64_MAX;
    MMB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    g_host_pool[dev] = pool;
  }
  *out = g_host_pool[dev];
  return MMB_OK;
}

struct DevBuf {
  void* p = nullptr;
  cudaStream_t st = nullptr;
  int alloc(size_t bytes, cudaStream_t s) {
    st = s;
    cudaMemPool_t pool;
    int rc = host_pool(&pool);
    if (rc) return rc;
    MMB_CUDA(cudaMallocFromPoolAsync(&p, bytes ? bytes : 16, pool, s));
    return MMB_OK;
  }
  ~DevBuf() {
    if (p) cudaFreeAsync(p, st);
  }
};
struct Streams {
  cudaStream_t in = nullptr, comp = nullptr, out = nullptr;
  std::vector<cudaEvent_t> ev;
  int init() {
    MMB_CUDA(cudaStreamCreateWithFlags(&in, cudaStreamNonBlocking));
    MMB_CUDA(cudaStreamCreateWithFlags(&comp, cudaStreamNonBlocking));
    MMB_CUDA(cudaStreamCreateWithFlags(&out, cudaStreamNonBlocking));
    return MMB_OK;
  }
  int event(cudaEvent_t* e) {
    MMB_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    ev.push_back(*e);
    return MMB_OK;
  }
  void sync_all() {
    if (in) cudaStreamSynchronize(in);
    if (out) cudaStreamSynchronize(out);
    if (comp) cudaStreamSynchronize(comp);
  }
  ~Streams() {
    for (auto e : ev) cudaEventDestroy(e);
    if (in) cudaStreamDestroy(in);
    if (comp) cudaStreamDestroy(comp);
    if (out) cudaStreamDestroy(out);
  }
};
}  // namespace

// Exchange parameters of the multi-GPU variant (world == 1: no exchange).
struct HostComm {
  int rank = 0, world = 1;
  void* const* bufs = nullptr;
  uint64_t epoch = 0;
  int64_t n_global = 0;
};

namespace {
// Declared AFTER the device buffers, hence destroyed BEFORE them: on every return path -- the early
// error returns included -- copies still in flight on the H2D / D2H streams finish before the buffers
// they use go back to the pool.
struct SyncGuard {
  Streams& S;
  ~SyncGuard() { S.sync_all(); }
};
// Multi-GPU: a rank that fails before it has enqueued the exchange tells its peers (abort flag) instead
// of letting them spin until the 4 s timeout.  Destroyed before SyncGuard, so the abort is synchronised too.
struct AbortGuard {
  const HostComm& hc;
  cudaStream_t st;
  bool armed;
  ~AbortGuard() {
    if (armed) mmb_comm_abort(hc.rank, hc.world, hc.bufs, hc.epoch, (mmb_stream_t)st);
  }
};

// Rows per chunk of a *_host call: 2^18 by default (chunk_rows <= 0), at most N.
int64_t host_chunk_rows(int64_t chunk_rows, int64_t N) {
  if (chunk_rows <= 0) chunk_rows = 1 << 18;
  if (chunk_rows > N) chunk_rows = N > 0 ? N : 1;
  return chunk_rows;
}

// The copy streams start once the allocations and uploads enqueued on `comp` so far are done.
int copy_streams_after_setup(Streams& S) {
  cudaEvent_t allocs_done;
  int rc = S.event(&allocs_done);
  if (rc) return rc;
  MMB_CUDA(cudaEventRecord(allocs_done, S.comp));
  MMB_CUDA(cudaStreamWaitEvent(S.in, allocs_done, 0));
  MMB_CUDA(cudaStreamWaitEvent(S.out, allocs_done, 0));
  return MMB_OK;
}

// Phase 1 of the *_host calls: the ids H2D in chunks of chunk_rows utterances (stream `in`, the two id buffers in
// turn) overlapped with the embed of the previous chunk (stream `comp`).  Per chunk, embed(ids_dev, r0, rows)
// enqueues the embed on `comp`; once its id buffer is free again, after(c, r0, rows) enqueues what else the chunk
// needs there.
template <class Embed, class After>
int stream_ids_in(Streams& S, DevBuf (&ids)[2], const int64_t* x_host, int64_t N, int64_t L, int64_t chunk_rows,
                  Embed&& embed, After&& after) {
  cudaEvent_t in_ready[2], buf_free[2];
  int rc;
  for (int b = 0; b < 2; ++b) {
    if ((rc = S.event(&in_ready[b]))) return rc;
    if ((rc = S.event(&buf_free[b]))) return rc;
  }
  const int64_t nchunks = ceil_div(N, chunk_rows);
  for (int64_t c = 0; c < nchunks; ++c) {
    const int b = (int)(c & 1);
    const int64_t r0 = c * chunk_rows;
    const int64_t rows = (N - r0) < chunk_rows ? (N - r0) : chunk_rows;
    if (c >= 2) MMB_CUDA(cudaStreamWaitEvent(S.in, buf_free[b], 0));
    MMB_CUDA(cudaMemcpyAsync(ids[b].p, x_host + r0 * L, (size_t)rows * L * sizeof(int64_t),
                             cudaMemcpyHostToDevice, S.in));
    MMB_CUDA(cudaEventRecord(in_ready[b], S.in));
    MMB_CUDA(cudaStreamWaitEvent(S.comp, in_ready[b], 0));
    if ((rc = embed((const int64_t*)ids[b].p, r0, rows))) return rc;
    MMB_CUDA(cudaEventRecord(buf_free[b], S.comp));
    if ((rc = after(c, r0, rows))) return rc;
  }
  return MMB_OK;
}

// The end of a *_host call: the status word read back behind everything on `comp`, all three streams drained, and
// the status turned into its error code.
int finish_host_call(Streams& S, const DevBuf& status, int64_t V) {
  int h_status = 0;
  MMB_CUDA(cudaMemcpyAsync(&h_status, status.p, sizeof(int), cudaMemcpyDeviceToHost, S.comp));
  MMB_CUDA(cudaStreamSynchronize(S.comp));
  MMB_CUDA(cudaStreamSynchronize(S.out));
  MMB_CUDA(cudaStreamSynchronize(S.in));
  if (h_status & MMB_STATUS_COMM_TIMEOUT) {
    set_error("peer all-reduce timed out: a rank never raised its flag");
    return MMB_E_COMM;
  }
  if (h_status & MMB_STATUS_BAD_INDEX) {
    set_error("index out of bounds: a token id is outside [-%lld, %lld)", (long long)V, (long long)V);
    return MMB_E_INDEX;
  }
  return MMB_OK;
}

// The Gram of chunk c (rows of emb_chunk) added to the running sum G, in chunk order (deterministic): G is the
// first chunk's Gram, then G += each next one.  gchunk: d x d scratch.
int add_chunk_gram(const float* emb_chunk, int64_t rows, int d, int64_t c, float* G, float* gchunk, void* gram_ws,
                   size_t gram_ws_bytes, int gram_mode, cudaStream_t st) {
  int rc = mmb_gram(emb_chunk, rows, d, gchunk, gram_ws, gram_ws_bytes, gram_mode, st);
  if (rc) return rc;
  accumulate_kernel<<<(d * d + 255) / 256, 256, 0, st>>>(G, gchunk, d * d, c == 0);
  MMB_LAUNCH_CHECK("accumulate");
  return MMB_OK;
}

// The components from the Gram G of n_global rows, in the workspace layout of sif_ws_layout: the start block (X^T
// Omega when n_global < d, from the N rows of emb, which are then every row) and the solve into pc_dev.
int components_from_gram(const float* G, const float* emb, int64_t N, int64_t n_global, int d, int npc,
                         const double* omega_dev, char* ws_base, const SifWs& Lw, float* pc_dev, cudaStream_t st) {
  const int k = npc + 10;
  const double* S0 = omega_dev;
  const int transposed = n_global < d;
  if (transposed) {
    int rc = mmb_start_block_xt(emb, N, d, omega_dev, k, (double*)(ws_base + Lw.s0), st);
    if (rc) return rc;
    S0 = (const double*)(ws_base + Lw.s0);
  }
  return mmb_pc_from_gram(G, d, S0, k, npc, transposed, 7, pc_dev, ws_base + Lw.pc, Lw.s0 - Lw.pc, st);
}
}  // namespace

static int sif_embedding_host_impl(const float* table_dev, int64_t V, int d, const float* vocab_w_dev,
                                   const int64_t* x_host, int64_t N, int64_t L, int npc,
                                   const double* Omega_host, void* emb_host, int emb_f64,
                                   float* pc_host, int gram_mode, int64_t chunk_rows, const HostComm& hc) {
  MMB_REQUIRE(table_dev && vocab_w_dev && (x_host || N == 0) && (emb_host || N == 0), "null pointer");
  MMB_REQUIRE(N >= 0 && L >= 0 && d > 0 && d % 4 == 0, "bad size");
  MMB_REQUIRE(npc >= 0 && npc + 10 <= 32, "npc must be in [0, 22]");
  MMB_REQUIRE(npc == 0 || Omega_host, "Omega is required when npc > 0");
  const bool dist = hc.world > 1;
  const int64_t n_global = dist ? hc.n_global : N;
  MMB_REQUIRE(!dist || n_global >= d, "the multi-GPU host path needs N_global >= d (use sif_dist for tiny splits)");
  if (N == 0 && !(dist && npc > 0)) return MMB_OK;
  chunk_rows = host_chunk_rows(chunk_rows, N);
  const int64_t nchunks = ceil_div(N, chunk_rows);
  const int k = npc + 10;

  Streams S;
  int rc = S.init();
  if (rc) return rc;
  DevBuf ids[2], emb, ws, omega, status, pcv, f64[2], gchunk, scaled;
  SyncGuard sync_guard{S};
  AbortGuard abort_guard{hc, S.comp, dist && npc > 0};
  const bool chunked_gram = npc > 0 && nchunks > 1;
  const size_t ids_chunk = (size_t)chunk_rows * L * sizeof(int64_t);
  if ((rc = ids[0].alloc(ids_chunk, S.comp))) return rc;
  if ((rc = ids[1].alloc(ids_chunk, S.comp))) return rc;
  if ((rc = emb.alloc((size_t)(N > 0 ? N : 1) * d * sizeof(float), S.comp))) return rc;
  if ((rc = status.alloc(sizeof(int), S.comp))) return rc;
  MMB_CUDA(cudaMemsetAsync(status.p, 0, sizeof(int), S.comp));
  const size_t ws_bytes = mmb_sif_workspace_bytes(N > 0 ? N : 1, d, npc);
  if (npc > 0) {
    const int64_t orows = n_global >= d ? d : N;
    if ((rc = ws.alloc(ws_bytes, S.comp))) return rc;
    if ((rc = omega.alloc((size_t)orows * k * sizeof(double), S.comp))) return rc;
    if ((rc = pcv.alloc((size_t)npc * d * sizeof(float), S.comp))) return rc;
    if (chunked_gram && (rc = gchunk.alloc((size_t)d * d * sizeof(float), S.comp))) return rc;
    MMB_CUDA(cudaMemcpyAsync(omega.p, Omega_host, (size_t)orows * k * sizeof(double),
                             cudaMemcpyHostToDevice, S.comp));
  }
  if (emb_f64) {
    const size_t b = (size_t)chunk_rows * d * sizeof(double);
    if ((rc = f64[0].alloc(b, S.comp))) return rc;
    if ((rc = f64[1].alloc(b, S.comp))) return rc;
  }
  // large batches: weights folded into the table once (sif_embed.cu); decided on the WHOLE batch, not per chunk
  const size_t scaled_bytes = mmb_sif_embed_workspace_bytes(V, d, N, L);
  if (scaled_bytes) {
    if ((rc = scaled.alloc(scaled_bytes, S.comp))) return rc;
    if ((rc = sif_prescale(table_dev, V, d, vocab_w_dev, scaled.p, S.comp))) return rc;
  }
  if ((rc = copy_streams_after_setup(S))) return rc;

  // phase 1: ids H2D (stream `in`) overlapped with the embed kernel (stream `comp`)
  rc = stream_ids_in(
      S, ids, x_host, N, L, chunk_rows,
      [&](const int64_t* ids_dev, int64_t r0, int64_t rows) {
        if (scaled_bytes)
          return sif_embed_prescaled(table_dev, V, d, vocab_w_dev, scaled.p, ids_dev, rows, L,
                                     (float*)emb.p + r0 * d, (int*)status.p, S.comp);
        return mmb_sif_embed(table_dev, V, d, vocab_w_dev, ids_dev, rows, L, (float*)emb.p + r0 * d,
                             (int*)status.p, S.comp);
      },
      [&](int64_t c, int64_t r0, int64_t rows) {
        if (!chunked_gram) return (int)MMB_OK;
        // The compute stream idles while the next chunk's ids cross PCIe: take the chunk's Gram now
        // and add it to the running sum, so that only the component solve separates the last H2D
        // from the first D2H.
        SifWs Lw = sif_ws_layout(N, d, npc);
        char* base = (char*)ws.p;
        return add_chunk_gram((const float*)emb.p + r0 * d, rows, d, c, (float*)(base + Lw.G), (float*)gchunk.p,
                              base + Lw.gram, Lw.pc - Lw.gram, gram_mode, S.comp);
      });
  if (rc) return rc;
  // phase 2: components from the Gram of the whole block (summed per chunk above, or taken here)
  float* pc_dev = (float*)pcv.p;
  if (npc > 0) {
    SifWs Lw = sif_ws_layout(N > 0 ? N : 1, d, npc);
    char* base = (char*)ws.p;
    float* G = (float*)(base + Lw.G);
    if (!chunked_gram) {
      if (N > 0) {
        rc = mmb_gram((const float*)emb.p, N, d, G, base + Lw.gram, Lw.pc - Lw.gram, gram_mode, S.comp);
        if (rc) return rc;
      } else {
        MMB_CUDA(cudaMemsetAsync(G, 0, (size_t)d * d * sizeof(float), S.comp));
      }
    }
    if (dist) {   // sum of the ranks' Grams over NVLink peer memory, rank order -> identical bits
      rc = mmb_allreduce_peer(G, (int64_t)d * d, 0, hc.rank, hc.world, hc.bufs, hc.epoch, (int*)status.p,
                              (mmb_stream_t)S.comp);
      if (rc) return rc;
      abort_guard.armed = false;   // this rank has taken part in the exchange
    }
    rc = components_from_gram(G, (const float*)emb.p, N, n_global, d, npc, (const double*)omega.p, base, Lw, pc_dev,
                              S.comp);
    if (rc) return rc;
  }
  // phase 3: projection (stream `comp`) overlapped with the D2H of finished chunks (`out`)
  cudaEvent_t out_ready[2], out_free[2];
  for (int b = 0; b < 2; ++b) {
    if ((rc = S.event(&out_ready[b]))) return rc;
    if ((rc = S.event(&out_free[b]))) return rc;
  }
  for (int64_t c = 0; c < nchunks; ++c) {
    const int b = (int)(c & 1);
    const int64_t r0 = c * chunk_rows;
    const int64_t rows = (N - r0) < chunk_rows ? (N - r0) : chunk_rows;
    float* blk = (float*)emb.p + r0 * d;
    if (npc > 0) {
      rc = mmb_remove_pc(blk, rows, d, pc_dev, npc, blk, S.comp);
      if (rc) return rc;
    }
    if (emb_f64) {
      if (c >= 2) MMB_CUDA(cudaStreamWaitEvent(S.comp, out_free[b], 0));
      const int64_t n = rows * d;
      f32_to_f64_kernel<<<(int)(ceil_div(n, 1024) < 4096 ? ceil_div(n, 1024) : 4096), 256, 0, S.comp>>>(
          blk, (double*)f64[b].p, n);
      MMB_LAUNCH_CHECK("f32_to_f64");
    }
    MMB_CUDA(cudaEventRecord(out_ready[b], S.comp));
    MMB_CUDA(cudaStreamWaitEvent(S.out, out_ready[b], 0));
    if (emb_f64) {
      MMB_CUDA(cudaMemcpyAsync((double*)emb_host + r0 * d, f64[b].p, (size_t)rows * d * sizeof(double),
                               cudaMemcpyDeviceToHost, S.out));
      MMB_CUDA(cudaEventRecord(out_free[b], S.out));
    } else {
      MMB_CUDA(cudaMemcpyAsync((float*)emb_host + r0 * d, blk, (size_t)rows * d * sizeof(float),
                               cudaMemcpyDeviceToHost, S.out));
    }
  }
  if (pc_host && npc > 0)
    MMB_CUDA(cudaMemcpyAsync(pc_host, pc_dev, (size_t)npc * d * sizeof(float), cudaMemcpyDeviceToHost, S.comp));
  return finish_host_call(S, status, V);
}

extern "C" int mmb_host_pipeline_trim(size_t keep_bytes) {
  int dev = 0;
  MMB_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && g_host_pool[dev]) MMB_CUDA(cudaMemPoolTrimTo(g_host_pool[dev], keep_bytes));
  return MMB_OK;
}

extern "C" int mmb_sif_embedding_host(const float* table_dev, int64_t V, int d, const float* vocab_w_dev,
                                      const int64_t* x_host, int64_t N, int64_t L, int npc,
                                      const double* Omega_host, void* emb_host, int emb_f64,
                                      float* pc_host, int gram_mode, int64_t chunk_rows) {
  return sif_embedding_host_impl(table_dev, V, d, vocab_w_dev, x_host, N, L, npc, Omega_host, emb_host, emb_f64,
                                 pc_host, gram_mode, chunk_rows, HostComm());
}

extern "C" int mmb_sif_embedding_host_peer(const float* table_dev, int64_t V, int d, const float* vocab_w_dev,
                                           const int64_t* x_host, int64_t N_local, int64_t L, int npc,
                                           const double* Omega_host, void* emb_host, int emb_f64,
                                           float* pc_host, int gram_mode, int64_t chunk_rows, int64_t N_global,
                                           int rank, int world, void* const* bufs, uint64_t epoch) {
  MMB_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank / world");
  MMB_REQUIRE(world == 1 || (bufs && epoch > 0), "exchange buffers and epoch > 0 are required");
  HostComm hc;
  hc.rank = rank; hc.world = world; hc.bufs = bufs; hc.epoch = epoch; hc.n_global = N_global;
  return sif_embedding_host_impl(table_dev, V, d, vocab_w_dev, x_host, N_local, L, npc, Omega_host, emb_host,
                                 emb_f64, pc_host, gram_mode, chunk_rows, hc);
}

// ---- the SIF sweep with host buffers ------------------------------------------------------------
// One staging buffer of the projection holds at most this many bytes, whatever P is.
static constexpr size_t kSweepStageBytes = (size_t)256 << 20;

extern "C" int mmb_sif_embedding_sweep_host(const float* table_dev, int64_t V, int d, const float* W_dev, int K,
                                            const int64_t* x_host, int64_t N, int64_t L, int P, const int* npcs,
                                            const double* const* Omega_host, void* out_host, int out_f64,
                                            int gram_mode, int64_t chunk_rows) {
  MMB_REQUIRE(table_dev && W_dev && npcs && (x_host || N == 0) && (out_host || N == 0), "null pointer");
  MMB_REQUIRE(N >= 0 && L >= 0 && d > 0 && d % 4 == 0 && d <= 1024, "bad size (d must be a multiple of 4, <= 1024)");
  MMB_REQUIRE(V > 0 && V < (int64_t)1 << 31, "V out of range");
  MMB_REQUIRE(K >= 1, "K must be >= 1");
  MMB_REQUIRE(P >= 1, "P must be >= 1");
  MMB_REQUIRE((uintptr_t)table_dev % 16 == 0, "table must be 16-byte aligned");
  bool any_pc = false;
  int npc_sum = 0;
  for (int j = 0; j < P; ++j) {
    MMB_REQUIRE(npcs[j] >= 0 && npcs[j] + 10 <= 32, "npc must be in [0, 22]");
    MMB_REQUIRE(npcs[j] == 0 || (Omega_host && Omega_host[j]), "Omega is required when npc > 0");
    any_pc |= npcs[j] > 0;
    npc_sum += npcs[j];
  }
  if (N == 0) return MMB_OK;
  chunk_rows = host_chunk_rows(chunk_rows, N);
  const size_t esz = out_f64 ? sizeof(double) : sizeof(float);
  // projection chunks: at most chunk_rows rows, and P rows of output per row within one staging buffer
  const size_t prow_bytes = (size_t)P * d * esz;
  int64_t out_rows = (int64_t)(kSweepStageBytes / prow_bytes);
  if (out_rows < 1) out_rows = 1;
  if (out_rows > chunk_rows) out_rows = chunk_rows;
  const bool transposed = N < d;
  const int64_t orows = transposed ? N : d;

  Streams S;
  int rc = S.init();
  if (rc) return rc;
  DevBuf ids[2], emb, wsm, status, G, gws, pcws, s0, pcv, omega, stage[2];
  SyncGuard sync_guard{S};
  const size_t ids_chunk = (size_t)chunk_rows * L * sizeof(int64_t);
  if ((rc = ids[0].alloc(ids_chunk, S.comp))) return rc;
  if ((rc = ids[1].alloc(ids_chunk, S.comp))) return rc;
  if ((rc = emb.alloc((size_t)K * N * d * sizeof(float), S.comp))) return rc;
  const size_t wsm_bytes = mmb_sif_embed_multi_workspace_bytes(V, K);
  if ((rc = wsm.alloc(wsm_bytes, S.comp))) return rc;
  if ((rc = status.alloc(sizeof(int), S.comp))) return rc;
  MMB_CUDA(cudaMemsetAsync(status.p, 0, sizeof(int), S.comp));
  for (int b = 0; b < 2; ++b)
    if ((rc = stage[b].alloc((size_t)out_rows * prow_bytes, S.comp))) return rc;
  // components: one Gram at a time, the P start blocks (uploaded once), the npc_sum rows of one k's components
  std::vector<size_t> omega_off(P, 0), pc_off(P, 0);
  size_t gws_bytes = 0, pcws_bytes = 0;
  if (any_pc) {
    size_t o = 0, q = 0;
    for (int j = 0; j < P; ++j) {
      omega_off[j] = o;
      pc_off[j] = q;
      if (!npcs[j]) continue;
      o += (size_t)orows * (npcs[j] + 10);
      q += (size_t)npcs[j] * d;
      const size_t b = mmb_pc_workspace_bytes(d, npcs[j] + 10);
      if (b > pcws_bytes) pcws_bytes = b;
    }
    gws_bytes = mmb_gram_workspace_bytes(N, d, gram_mode);
    if ((rc = G.alloc((size_t)d * d * sizeof(float), S.comp))) return rc;
    if ((rc = gws.alloc(gws_bytes, S.comp))) return rc;
    if ((rc = pcws.alloc(pcws_bytes, S.comp))) return rc;
    if ((rc = pcv.alloc(q * sizeof(float), S.comp))) return rc;
    if ((rc = omega.alloc(o * sizeof(double), S.comp))) return rc;
    if (transposed && (rc = s0.alloc((size_t)d * 32 * sizeof(double), S.comp))) return rc;
    for (int j = 0; j < P; ++j)
      if (npcs[j])
        MMB_CUDA(cudaMemcpyAsync((double*)omega.p + omega_off[j], Omega_host[j],
                                 (size_t)orows * (npcs[j] + 10) * sizeof(double), cudaMemcpyHostToDevice, S.comp));
  }
  if ((rc = sif_embed_multi_weights(W_dev, V, d, K, wsm.p, S.comp))) return rc;
  if ((rc = copy_streams_after_setup(S))) return rc;

  // phase 1: ids H2D (stream `in`) overlapped with the K-vector embed (stream `comp`) into the resident emb
  float* E0 = (float*)emb.p;
  rc = stream_ids_in(
      S, ids, x_host, N, L, chunk_rows,
      [&](const int64_t* ids_dev, int64_t r0, int64_t rows) {
        return sif_embed_multi_chunk(table_dev, V, d, wsm.p, K, ids_dev, rows, L, N, E0 + r0 * d, (int*)status.p,
                                     S.comp);
      },
      [](int64_t, int64_t, int64_t) { return (int)MMB_OK; });
  if (rc) return rc;

  // phases 2 and 3 per k: the Gram of the whole emb[k] and its components (as the device sweep takes them), then
  // the projection of each chunk into a staging buffer (stream `comp`) overlapped with the D2H of the previous
  // chunk (stream `out`); the next k's Gram runs while the last chunk of this k crosses PCIe
  cudaEvent_t out_ready[2], out_free[2];
  for (int b = 0; b < 2; ++b) {
    if ((rc = S.event(&out_ready[b]))) return rc;
    if ((rc = S.event(&out_free[b]))) return rc;
  }
  std::vector<const float*> pcs(P, nullptr);
  std::vector<void*> outs(P, nullptr);
  int64_t q = 0;                   // chunks projected so far, over all k
  int64_t pend_k = 0, pend_r0 = 0, pend_rows = 0;
  // the D2H of projected chunk q - 1: P copies from its staging buffer into out_host[k, j, r0 : r0 + rows]
  auto copy_out = [&](int64_t qq, int64_t k, int64_t r0, int64_t rows) {
    const int b = (int)(qq & 1);
    MMB_CUDA(cudaStreamWaitEvent(S.out, out_ready[b], 0));
    for (int j = 0; j < P; ++j)
      MMB_CUDA(cudaMemcpyAsync((char*)out_host + (((size_t)k * P + j) * N + r0) * d * esz,
                               (char*)stage[b].p + (size_t)j * rows * d * esz, (size_t)rows * d * esz,
                               cudaMemcpyDeviceToHost, S.out));
    MMB_CUDA(cudaEventRecord(out_free[b], S.out));
    return (int)MMB_OK;
  };
  for (int k = 0; k < K; ++k) {
    const float* E = E0 + (size_t)k * N * d;
    if (any_pc) {
      if ((rc = mmb_gram(E, N, d, (float*)G.p, gws.p, gws_bytes, gram_mode, S.comp))) return rc;
      for (int j = 0; j < P; ++j) {
        if (!npcs[j]) continue;
        const int kk = npcs[j] + 10;
        const double* S0 = (const double*)omega.p + omega_off[j];
        if (transposed) {
          if ((rc = mmb_start_block_xt(E, N, d, S0, kk, (double*)s0.p, S.comp))) return rc;
          S0 = (const double*)s0.p;
        }
        float* pc = (float*)pcv.p + pc_off[j];
        rc = mmb_pc_from_gram((const float*)G.p, d, S0, kk, npcs[j], transposed, 7, pc, pcws.p, pcws_bytes, S.comp);
        if (rc) return rc;
        pcs[j] = pc;
      }
    }
    for (int64_t r0 = 0; r0 < N; r0 += out_rows, ++q) {
      const int64_t rows = (N - r0) < out_rows ? (N - r0) : out_rows;
      const int b = (int)(q & 1);
      if (q >= 2) MMB_CUDA(cudaStreamWaitEvent(S.comp, out_free[b], 0));
      for (int j = 0; j < P; ++j) outs[j] = (char*)stage[b].p + (size_t)j * rows * d * esz;
      rc = remove_pc_multi(E + r0 * d, rows, d, P, pcs.data(), npcs, outs.data(), out_f64 != 0, S.comp);
      if (rc) return rc;
      MMB_CUDA(cudaEventRecord(out_ready[b], S.comp));
      // enqueued after this chunk's projection, so that a D2H into pageable memory (which returns only when
      // done) still overlaps it
      if (q > 0 && (rc = copy_out(q - 1, pend_k, pend_r0, pend_rows))) return rc;
      pend_k = k; pend_r0 = r0; pend_rows = rows;
    }
  }
  if ((rc = copy_out(q - 1, pend_k, pend_r0, pend_rows))) return rc;
  return finish_host_call(S, status, V);
}

// ---- SIF fit / transform with host buffers -----------------------------------------------------------------
extern "C" int mmb_sif_transform_host(const float* table_dev, int64_t V, int d, const float* vocab_w_dev,
                                      const int64_t* x_host, int64_t N, int64_t L, const float* pc_host, int npc,
                                      void* out_host, int out_f64, int64_t chunk_rows) {
  MMB_REQUIRE(table_dev && vocab_w_dev && (x_host || N == 0) && (out_host || N == 0), "null pointer");
  MMB_REQUIRE(N >= 0 && L >= 0 && d > 0 && d % 4 == 0 && d <= 1024, "bad size (d must be a multiple of 4, <= 1024)");
  MMB_REQUIRE(npc >= 0 && npc <= 32, "npc must be in [0, 32]");
  MMB_REQUIRE(pc_host || npc == 0, "null pointer");
  if (N == 0) return MMB_OK;
  chunk_rows = host_chunk_rows(chunk_rows, N);
  const size_t esz = out_f64 ? sizeof(double) : sizeof(float);

  Streams S;
  int rc = S.init();
  if (rc) return rc;
  DevBuf ids[2], stage[2], status, pcv, scaled;
  SyncGuard sync_guard{S};
  const size_t ids_chunk = (size_t)chunk_rows * L * sizeof(int64_t);
  for (int b = 0; b < 2; ++b) {
    if ((rc = ids[b].alloc(ids_chunk, S.comp))) return rc;
    if ((rc = stage[b].alloc((size_t)chunk_rows * d * esz, S.comp))) return rc;
  }
  if ((rc = status.alloc(sizeof(int), S.comp))) return rc;
  MMB_CUDA(cudaMemsetAsync(status.p, 0, sizeof(int), S.comp));
  if (npc > 0) {
    if ((rc = pcv.alloc((size_t)npc * d * sizeof(float), S.comp))) return rc;
    MMB_CUDA(cudaMemcpyAsync(pcv.p, pc_host, (size_t)npc * d * sizeof(float), cudaMemcpyHostToDevice, S.comp));
  }
  // the kernel variant of the WHOLE batch: the pre-scaled table once, and N as the CTA-per-utterance rule's N
  const size_t scaled_bytes = mmb_sif_embed_workspace_bytes(V, d, N, L);
  if (scaled_bytes) {
    if ((rc = scaled.alloc(scaled_bytes, S.comp))) return rc;
    if ((rc = sif_prescale(table_dev, V, d, vocab_w_dev, scaled.p, S.comp))) return rc;
  }
  if ((rc = copy_streams_after_setup(S))) return rc;

  // ids H2D (stream `in`) || the fused embed + projection of a chunk into a staging buffer (`comp`) || the D2H of the
  // previous chunk (`out`): nothing depends on the whole batch, so the three run at once
  cudaEvent_t out_ready[2], out_free[2];
  for (int b = 0; b < 2; ++b) {
    if ((rc = S.event(&out_ready[b]))) return rc;
    if ((rc = S.event(&out_free[b]))) return rc;
  }
  auto copy_out = [&](int64_t c) {
    const int b = (int)(c & 1);
    const int64_t r0 = c * chunk_rows;
    const int64_t rows = (N - r0) < chunk_rows ? (N - r0) : chunk_rows;
    MMB_CUDA(cudaStreamWaitEvent(S.out, out_ready[b], 0));
    MMB_CUDA(cudaMemcpyAsync((char*)out_host + (size_t)r0 * d * esz, stage[b].p, (size_t)rows * d * esz,
                             cudaMemcpyDeviceToHost, S.out));
    MMB_CUDA(cudaEventRecord(out_free[b], S.out));
    return (int)MMB_OK;
  };
  rc = stream_ids_in(
      S, ids, x_host, N, L, chunk_rows,
      [&](const int64_t* ids_dev, int64_t r0, int64_t rows) {
        const int64_t c = r0 / chunk_rows;
        const int b = (int)(c & 1);
        if (c >= 2) MMB_CUDA(cudaStreamWaitEvent(S.comp, out_free[b], 0));
        return sif_transform_chunk(table_dev, V, d, vocab_w_dev, scaled_bytes ? scaled.p : nullptr, ids_dev, rows, L,
                                   N, (const float*)pcv.p, npc, stage[b].p, out_f64 != 0, (int*)status.p, S.comp);
      },
      [&](int64_t c, int64_t, int64_t) {
        MMB_CUDA(cudaEventRecord(out_ready[c & 1], S.comp));
        // the D2H of the previous chunk, enqueued after this chunk's kernel, so that a copy into pageable memory
        // (which returns only when done) still overlaps it
        return c > 0 ? copy_out(c - 1) : (int)MMB_OK;
      });
  if (rc) return rc;
  if ((rc = copy_out(ceil_div(N, chunk_rows) - 1))) return rc;
  return finish_host_call(S, status, V);
}

extern "C" int mmb_sif_fit_host(const float* table_dev, int64_t V, int d, const float* vocab_w_dev,
                                const int64_t* x_host, int64_t N, int64_t L, int npc, const double* Omega_host,
                                float* pc_host, int gram_mode, int64_t chunk_rows) {
  MMB_REQUIRE(table_dev && vocab_w_dev && x_host && Omega_host && pc_host, "null pointer");
  MMB_REQUIRE(N >= 1 && L >= 0 && d > 0 && d % 4 == 0 && d <= 512,
              "bad size (N >= 1; d must be a multiple of 4, <= 512)");
  MMB_REQUIRE(npc >= 1 && npc + 10 <= 32, "npc must be in [1, 22]");
  // N < d: the start block X^T Omega needs every row at once
  chunk_rows = N < d ? N : host_chunk_rows(chunk_rows, N);
  const int64_t nchunks = ceil_div(N, chunk_rows);
  const int k = npc + 10;
  const int64_t orows = N >= d ? d : N;

  Streams S;
  int rc = S.init();
  if (rc) return rc;
  DevBuf ids[2], emb, ws, omega, status, pcv, gchunk, scaled;
  SyncGuard sync_guard{S};
  const size_t ids_chunk = (size_t)chunk_rows * L * sizeof(int64_t);
  if ((rc = ids[0].alloc(ids_chunk, S.comp))) return rc;
  if ((rc = ids[1].alloc(ids_chunk, S.comp))) return rc;
  if ((rc = emb.alloc((size_t)chunk_rows * d * sizeof(float), S.comp))) return rc;
  if ((rc = status.alloc(sizeof(int), S.comp))) return rc;
  MMB_CUDA(cudaMemsetAsync(status.p, 0, sizeof(int), S.comp));
  const SifWs Lw = sif_ws_layout(N, d, npc);
  if ((rc = ws.alloc(Lw.total, S.comp))) return rc;
  if ((rc = omega.alloc((size_t)orows * k * sizeof(double), S.comp))) return rc;
  if ((rc = pcv.alloc((size_t)npc * d * sizeof(float), S.comp))) return rc;
  if (nchunks > 1 && (rc = gchunk.alloc((size_t)d * d * sizeof(float), S.comp))) return rc;
  MMB_CUDA(cudaMemcpyAsync(omega.p, Omega_host, (size_t)orows * k * sizeof(double), cudaMemcpyHostToDevice, S.comp));
  const size_t scaled_bytes = mmb_sif_embed_workspace_bytes(V, d, N, L);
  if (scaled_bytes) {
    if ((rc = scaled.alloc(scaled_bytes, S.comp))) return rc;
    if ((rc = sif_prescale(table_dev, V, d, vocab_w_dev, scaled.p, S.comp))) return rc;
  }
  if ((rc = copy_streams_after_setup(S))) return rc;

  // ids H2D (stream `in`) || embed of a chunk, then its Gram added to the running sum (`comp`); one embedding chunk
  // suffices because the Gram of chunk c runs on `comp` before the embed of chunk c + 1
  char* base = (char*)ws.p;
  float* G = (float*)(base + Lw.G);
  rc = stream_ids_in(
      S, ids, x_host, N, L, chunk_rows,
      [&](const int64_t* ids_dev, int64_t, int64_t rows) {
        return sif_transform_chunk(table_dev, V, d, vocab_w_dev, scaled_bytes ? scaled.p : nullptr, ids_dev, rows, L,
                                   N, nullptr, 0, emb.p, false, (int*)status.p, S.comp);
      },
      [&](int64_t c, int64_t, int64_t rows) {
        if (nchunks == 1)
          return mmb_gram((const float*)emb.p, rows, d, G, base + Lw.gram, Lw.pc - Lw.gram, gram_mode, S.comp);
        return add_chunk_gram((const float*)emb.p, rows, d, c, G, (float*)gchunk.p, base + Lw.gram, Lw.pc - Lw.gram,
                              gram_mode, S.comp);
      });
  if (rc) return rc;
  rc = components_from_gram(G, (const float*)emb.p, N, N, d, npc, (const double*)omega.p, base, Lw, (float*)pcv.p,
                            S.comp);
  if (rc) return rc;
  MMB_CUDA(cudaMemcpyAsync(pc_host, pcv.p, (size_t)npc * d * sizeof(float), cudaMemcpyDeviceToHost, S.comp));
  return finish_host_call(S, status, V);
}
