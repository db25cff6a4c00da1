/*
 * mmb_b200.h -- C ABI of libmmb_b200.so, the sm_100a implementation of the SIF / MMB
 * utterance-embedding hot path of yaochie/multimodal-baselines.
 *
 * The reference has no FFI of its own (pure Python); the boundary is the module-level
 * Python API of sif_functions.py / sif.py / losses.py / models.py / simplesif.py
 * (SURVEY.md section 8b).  Every entry point below names the reference function
 * (file:line under the reference tree) whose arithmetic it replaces.  The Python shims in
 * multimodal-baselines_b200/ bind these with ctypes (see INTEGRATION.md) and keep the
 * reference's names, argument order and error behaviour.
 *
 * Conventions
 *   - plain C types only; all "device" pointers are CUDA device pointers owned by the
 *     caller (torch allocates them); the library allocates nothing persistent except in
 *     the *_host entry points, which own their staging buffers for the call's duration;
 *   - every launch goes to the cudaStream_t passed as `stream` (0 = legacy default) and
 *     returns without synchronising unless stated otherwise;
 *   - return value 0 = success; non-zero = MMB_E_* below, message in mmb_last_error();
 *   - matrices are row-major and dense unless a leading dimension is given;
 *   - `status` words are device ints the kernels OR error bits into (MMB_STATUS_*); the
 *     caller zeroes them, and reads them back when it next synchronises.
 */
#ifndef MMB_B200_H
#define MMB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* mmb_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define MMB_API __attribute__((visibility("default")))
#else
#define MMB_API
#endif

enum {
  MMB_OK = 0,
  MMB_E_INVALID = 1,     /* bad argument (null pointer, unsupported size)            */
  MMB_E_CUDA = 2,        /* a CUDA runtime call failed; see mmb_last_error()         */
  MMB_E_UNSUPPORTED = 3, /* valid request this build / device cannot run             */
  MMB_E_INDEX = 4,       /* token id outside [-V, V): the reference's IndexError      */
  MMB_E_COMM = 5         /* a peer rank never arrived in a *_peer call (timeout)      */
};

enum {
  MMB_STATUS_BAD_INDEX = 1, /* an id was outside [-V, V) (NumPy would raise IndexError) */
  MMB_STATUS_NONFINITE = 2, /* a log-probability was +-inf/NaN (losses.py:258-264)      */
  MMB_STATUS_COMM_TIMEOUT = 4 /* a peer never raised its flag in mmb_*_peer (rank died)   */
};

enum { /* mmb_gram `mode` */
  MMB_GRAM_AUTO = 0,
  MMB_GRAM_FP32 = 1,     /* CUDA-core FP32 FMA, split-K, deterministic 2-stage reduce  */
  MMB_GRAM_TF32X3 = 2    /* tcgen05 kind::tf32, 3xTF32 split (hi*hi + hi*lo + lo*hi)   */
};

/* ---------------------------------------------------------------- library --------- */
MMB_API int mmb_version(void);
MMB_API const char* mmb_last_error(void);
/* sm_count / cc_major / cc_minor of the current device (any pointer may be NULL). */
MMB_API int mmb_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* Instrumentation (no reference counterpart): number of kernels this library has launched in
 * this process so far (every launch site counts itself), and the template-expanded name of the
 * kernel a run-time dispatch chose last (tag 0 = the embed kernel of mmb_sif_embed /
 * mmb_weighted_average).  bench.py derives `gpu_launches` and `roofline.kernel` from these. */
MMB_API unsigned long long mmb_launch_count(void);
MMB_API const char* mmb_last_kernel(int tag);
/* Pinned host memory for the *_host entry points and for e2e benchmarks. */
MMB_API int mmb_host_alloc(void** ptr, size_t bytes);
/* Write-combined pinned memory: for buffers the host only WRITES and the device reads (the ids of the
 * *_host entry points); not snooped by the CPU caches on its way over PCIe, slow for host reads. */
MMB_API int mmb_host_alloc_wc(void** ptr, size_t bytes);
MMB_API int mmb_host_free(void* ptr);

/* ---------------------------------------------------------------- SIF (A1-A5) ----- */

/* seq2weight -- sif_functions.py:8-15.
 * w[i,j] = weight4ind[seq[i,j]] if (mask == NULL || mask[i,j] > 0) && seq[i,j] >= 0, else 0.
 * weight4ind is the float32 image of the reference's float64 vector (the reference casts
 * on assignment into its float32 array, line 9/13).  ids >= V set MMB_STATUS_BAD_INDEX. */
MMB_API int mmb_seq2weight(const int64_t* seq, const float* mask, const float* weight4ind, int64_t V,
                   int64_t N, int64_t L, float* w, int* status, mmb_stream_t stream);

/* get_weighted_average -- sif_functions.py:28-56 with explicit per-token weights.
 * emb[i,:] = (sum_j w[i,j] * table[x[i,j],:]) / count_nonzero(w[i,:]); negative ids index
 * from the end of the table as NumPy does; FP32 accumulate in token order.            */
MMB_API int mmb_weighted_average(const float* table, int64_t V, int d, const int64_t* x, const float* w,
                         int64_t N, int64_t L, float* emb, int* status, mmb_stream_t stream);

/* seq2weight (mask of ones, sif.py:78-82) fused into get_weighted_average: the (N,L)
 * weight matrix never exists.  w[i,j] = vocab_w[x[i,j]] if x[i,j] >= 0 else 0.         */
MMB_API int mmb_sif_embed(const float* table, int64_t V, int d, const float* vocab_w, const int64_t* x,
                  int64_t N, int64_t L, float* emb, int* status, mmb_stream_t stream);

/* mmb_sif_embed with scratch: for large batches (N * L >= 8 V) the vocabulary weights are folded into a
 * scratch copy of the table once per call (T' = w * T), after which a token costs one row read and one warp
 * shuffle -- no weight gather.  Same result up to one rounding per term (w * row rounded before the sum).
 * mmb_sif_embed_workspace_bytes returns 0 when the plain kernel is the right one (small batch, few long
 * rows, d > 512, table >= 4 GiB); with ws == NULL or too small the call IS mmb_sif_embed.              */
MMB_API size_t mmb_sif_embed_workspace_bytes(int64_t V, int d, int64_t N, int64_t L);
MMB_API int mmb_sif_embed_ws(const float* table, int64_t V, int d, const float* vocab_w, const int64_t* x,
                             int64_t N, int64_t L, float* emb, int* status, void* ws, size_t ws_bytes,
                             mmb_stream_t stream);

/* SIF embedding with GIVEN components (TruncatedSVD.transform's counterpart of compute_pc's fit: remove_pc,
 * sif_functions.py:69-81, with pc fitted elsewhere): mmb_sif_embed_ws (ws as there; NULL -> the general kernel)
 * followed by mmb_remove_pc(pc, npc), in one pass, bit for bit -- the warp that finishes a row subtracts its
 * projection before the row is stored.  pc: npc x d float32 on the device, 16-byte aligned; npc in [0, 32]; npc = 0
 * is the plain embed.  out (N, d) float32, 16-byte aligned.  mmb_last_kernel(0) names the embed kernel, followed
 * by " +pc f32" when npc > 0 (with npc = 0 the plain kernel runs, under its plain name).                        */
MMB_API int mmb_sif_transform(const float* table, int64_t V, int d, const float* vocab_w, const int64_t* x,
                              int64_t N, int64_t L, const float* pc, int npc, float* out, int* status,
                              void* ws, size_t ws_bytes, mmb_stream_t stream);

/* SIF sweep: seq2weight + get_weighted_average (sif_functions.py:8-15, 28-56) for K vocabulary-weight vectors
 * over one gather of the table rows.  vocab_w is (K, V) row-major; emb is (K, N, d), so every emb[k] is a dense
 * (N, d) matrix that mmb_gram / mmb_remove_pc take as it is.  emb[k] is bit-identical to mmb_sif_embed with
 * vocab_w = vocab_w[k] (the general kernel, not the pre-scaled one of mmb_sif_embed_ws): the same variant rule,
 * duplicate-row merging, summation order and per-vector divisor count_nonzero(w_k[i, :]).  Negative ids wrap
 * and weigh 0 for every k; ids outside [-V, V) set MMB_STATUS_BAD_INDEX.  Rows are read once per group of up to
 * Kg vectors (Kg = 8 for d <= 256, 4 for d <= 512, 2 for d <= 1024); any K >= 1 runs as ceil(K / Kg) passes.
 * ws: mmb_sif_embed_multi_workspace_bytes(V, K) bytes, 32-byte aligned (the weights, laid out per token);
 * too small a ws is MMB_E_INVALID.  The kernel of the last call is mmb_last_kernel(1).                  */
MMB_API size_t mmb_sif_embed_multi_workspace_bytes(int64_t V, int K);
MMB_API int mmb_sif_embed_multi(const float* table, int64_t V, int d, const float* vocab_w, int K, const int64_t* x,
                                int64_t N, int64_t L, float* emb, int* status, void* ws, size_t ws_bytes,
                                mmb_stream_t stream);
/* mmb_sif_embed_multi on ragged (CSR) ids (tokens, offsets, L_pad, pad_id as for mmb_sif_embed_ragged below): emb
 * is (K, N, d) and emb[k] is bit-identical to mmb_sif_embed_ragged with vocab_w = vocab_w[k].  The pad run of each
 * utterance is added in closed form per k (n_pad * vocab_w[k][pad_id] * table[pad_id] to the sum, n_pad to the
 * divisor when that weight is non-zero), so padding is neither stored nor walked.  d <= 512.  The same workspace
 * (mmb_sif_embed_multi_workspace_bytes(V, K)) and variant rule (L_pad >= 256 and N < 16 SMs: a CTA per utterance)
 * as mmb_sif_embed_multi.  MMB_STATUS_BAD_INDEX: a token outside [-V, V), an utterance longer than L_pad, or a
 * pad_id outside [-V, V) where padding is present.  mmb_last_kernel(1) names a *_ragged_* kernel.          */
MMB_API int mmb_sif_embed_multi_ragged(const float* table, int64_t V, int d, const float* vocab_w, int K,
                                       const int64_t* tokens, const int64_t* offsets, int64_t N, int64_t L_pad,
                                       int64_t pad_id, float* emb, int* status, void* ws, size_t ws_bytes,
                                       mmb_stream_t stream);

/* Ragged (CSR) ids, SURVEY.md 8f N3 -- the same result as mmb_sif_embed on the right-padded (N, L_pad)
 * matrix the reference builds (utils.py:77-80; sif_functions.py:28-56), without walking the padding:
 * utterance i is tokens[offsets[i] .. offsets[i+1]) (int64, offsets has N + 1 entries) and is understood
 * to be followed by L_pad - length_i copies of `pad_id`, whose contribution the kernel adds in closed form
 * (n_pad * vocab_w[pad_id] * table[pad_id] to the sum; n_pad to the divisor when that weight is non-zero --
 * the reference's divisor counts every token of the padded row, sif_functions.py:55).
 * mmb_ids_lengths / mmb_ids_compact convert a padded device matrix: length_i = 1 + index of the last token
 * that is not pad_id (interior pad ids stay tokens); offsets = exclusive prefix sums (N + 1 entries);
 * tokens = the rows' prefixes back to back (offsets[N] entries: read it back to size the buffer).      */
MMB_API int mmb_sif_embed_ragged(const float* table, int64_t V, int d, const float* vocab_w,
                                 const int64_t* tokens, const int64_t* offsets, int64_t N, int64_t L_pad,
                                 int64_t pad_id, float* emb, int* status, mmb_stream_t stream);
MMB_API int mmb_ids_lengths(const int64_t* ids, int64_t N, int64_t L, int64_t pad_id, int64_t* lengths,
                            int64_t* offsets, mmb_stream_t stream);
MMB_API int mmb_ids_compact(const int64_t* ids, int64_t N, int64_t L, const int64_t* offsets, int64_t* tokens,
                            mmb_stream_t stream);

/* compute_pc part 1 -- sif_functions.py:58-67: G = X^T X (d x d, float32), no centring.
 * `ws` is scratch of at least mmb_gram_workspace_bytes(N, d, mode) bytes.             */
MMB_API size_t mmb_gram_workspace_bytes(int64_t N, int d, int mode);
MMB_API int mmb_gram(const float* X, int64_t N, int d, float* G, void* ws, size_t ws_bytes, int mode,
             mmb_stream_t stream);

/* compute_pc part 2: the components sklearn's TruncatedSVD(npc, n_iter=7, random_state=0)
 * returns, as a function of G and the seeded start block S0 (d x k, row-major float64,
 * k = npc + 10): S0 = RandomState(0).normal(size=(d,k)) when N >= d (transposed = 0), or
 * X^T RandomState(0).normal(size=(N,k)) when N < d (transposed = 1); see
 * oracle/sif_oracle.py:compute_pc_from_gram.  pc is (npc, d) float32, unit rows, largest
 * |entry| of each row positive (sklearn svd_flip, u_based_decision=False).  FP64, as a
 * chain of n_iter + 3 kernels on `stream`.  Needs 1 <= d <= 512 and 1 <= npc <= k <= 32.
 * `ws` is scratch of at least mmb_pc_workspace_bytes(d, k) bytes.                      */
MMB_API size_t mmb_pc_workspace_bytes(int d, int k);
MMB_API int mmb_pc_from_gram(const float* G, int d, const double* S0, int k, int npc, int transposed,
                     int n_iter, float* pc, void* ws, size_t ws_bytes, mmb_stream_t stream);
/* S0 for the N < d case: S0 = X^T Omega (Omega is N x k float64, row-major).            */
MMB_API int mmb_start_block_xt(const float* X, int64_t N, int d, const double* Omega, int k, double* S0,
                       mmb_stream_t stream);

/* remove_pc -- sif_functions.py:69-81 given the components:
 * out = X - (X pc^T) pc  (npc == 1: line 78; npc > 1: line 80).  out may alias X.      */
MMB_API int mmb_remove_pc(const float* X, int64_t N, int d, const float* pc, int npc, float* out,
                  mmb_stream_t stream);
/* mmb_remove_pc for P component sets against ONE read of X: out[j] = X - (X pc[j]^T) pc[j], each out[j]
 * bit-identical to mmb_remove_pc(X, pc[j], npc[j]); npc[j] = 0 copies X (pc[j] may then be NULL).
 * pc and out are HOST arrays of P DEVICE pointers (pc[j]: npc[j] x d, out[j]: N x d); npc is a HOST
 * array.  Any P >= 1: one launch per group of up to 8 consecutive sets whose components fit 128 KB of
 * shared memory.  out[j] may alias X only when P == 1.  N == 0 launches nothing (X, out[j] may be NULL). */
MMB_API int mmb_remove_pc_multi(const float* X, int64_t N, int d, int P, const float* const* pc, const int* npc,
                                float* const* out, mmb_stream_t stream);

/* get_sentence_embeddings -- sif.py:84-94 on ONE device, everything resident in HBM:
 * embed -> Gram -> components (npc, 0 = skip PC removal) -> projection, no host sync.
 * `Omega` is the seeded start block for this (N, npc) (d x k if N >= d else N x k).
 * `ws` >= mmb_sif_workspace_bytes(N, d, npc).  emb is (N, d) float32; pc (npc, d) and
 * G (d, d) are written when non-NULL outputs are given.                                */
MMB_API size_t mmb_sif_workspace_bytes(int64_t N, int d, int npc);
MMB_API int mmb_sif_embedding(const float* table, int64_t V, int d, const float* vocab_w,
                      const int64_t* x, int64_t N, int64_t L, int npc, const double* Omega,
                      float* emb, float* pc, float* G, void* ws, size_t ws_bytes, int gram_mode,
                      int* status, mmb_stream_t stream);

/* The same call with HOST buffers (ids, Omega in; emb out), as the reference's NumPy
 * caller sees it: H2D of the ids in chunks overlapped with the embed kernel, one Gram +
 * solve, projection overlapped with the D2H of the result.  `table_dev` / `vocab_w_dev`
 * stay on the device (upload once with cudaMemcpy / torch).  x_host and emb_host should be
 * pinned (mmb_host_alloc) for full PCIe rate.  emb_f64 != 0 writes float64 like the
 * reference's np.zeros((N,d)) (sif_functions.py:37), else float32.  Synchronous.       */
MMB_API int mmb_sif_embedding_host(const float* table_dev, int64_t V, int d, const float* vocab_w_dev,
                           const int64_t* x_host, int64_t N, int64_t L, int npc,
                           const double* Omega_host, void* emb_host, int emb_f64,
                           float* pc_host, int gram_mode, int64_t chunk_rows);

/* The SIF sweep (mmb_sif_embed_multi, then per k one Gram, per (k, npc) one component solve and per k one
 * mmb_remove_pc_multi) with HOST buffers, as get_sentence_embeddings_sweep's NumPy caller sees it: x_host (N, L) in,
 * out_host (K, P, N, d) out, float64 when out_f64 != 0 (each value the float32 result widened once), else float32.
 * W_dev is (K, V) float32 on the device.  npcs and Omega_host are HOST arrays of P entries: Omega_host[j] is the
 * seeded start block for npcs[j] (d x (npc + 10) when N >= d, N x (npc + 10) when N < d, float64), NULL when
 * npcs[j] == 0.  out[k, j] is bit-identical to the device sweep's out[k, j] at every chunk_rows:
 *   1. ids H2D in chunks of chunk_rows utterances (<= 0: 2^18), double-buffered, overlapped with the K-vector
 *      embed of each chunk into a resident (K, N, d) float32 tensor (variant rule taken on the whole N);
 *   2. per k one mmb_gram over the whole emb[k] (gram_mode resolved on N, as the device sweep does), then one
 *      mmb_pc_from_gram per npc != 0 (start block mmb_start_block_xt(emb[k]) when N < d);
 *   3. per k and chunk of at most chunk_rows rows, one projection writes all P sets from one read of the rows
 *      into a (P, rows, d) staging buffer of the output type (at most 256 MB, so rows shrink as P grows),
 *      overlapped with P plain D2H copies of the previous chunk into out_host[k, j, r0 : r1].
 * Device memory: K * N * d * 4 bytes, plus two id buffers, two staging buffers and the Gram / solve scratch,
 * none of which grows with P.  x_host and out_host should be pinned (mmb_host_alloc) for full PCIe rate.
 * Synchronous.  N == 0 returns at once; a bad id is MMB_E_INDEX once every stream has drained.            */
MMB_API int mmb_sif_embedding_sweep_host(const float* table_dev, int64_t V, int d, const float* W_dev, int K,
                                         const int64_t* x_host, int64_t N, int64_t L, int P, const int* npcs,
                                         const double* const* Omega_host, void* out_host, int out_f64,
                                         int gram_mode, int64_t chunk_rows);

/* mmb_sif_transform from host buffers: ids H2D || fused kernel || D2H, chunk by chunk (chunk_rows <= 0: 2^18),
 * with two id buffers and two staging buffers of the output type on the device and nothing of size N -- no row
 * depends on the whole batch, so chunk c + 1's ids cross H2D while chunk c is embedded and chunk c - 1 crosses D2H.
 * pc_host: npc x d float32 on the host, npc in [0, 32].  out_host (N, d): float64 when out_f64 != 0 (the float32
 * result widened once), else float32.  The kernel variant (pre-scaled, CTA per utterance, wide table) is decided
 * on the WHOLE N, as mmb_sif_embedding_sweep_host does, so the result equals mmb_sif_transform on all N rows (with
 * ws of mmb_sif_embed_workspace_bytes) at every chunk_rows.  Synchronous; a bad id is MMB_E_INDEX.  The kernel
 * name (mmb_last_kernel(0)) ends in " +pc f32" (npc > 0), " +pc f64" (float64 out, any npc) or nothing.      */
MMB_API int mmb_sif_transform_host(const float* table_dev, int64_t V, int d, const float* vocab_w_dev,
                                   const int64_t* x_host, int64_t N, int64_t L, const float* pc_host, int npc,
                                   void* out_host, int out_f64, int64_t chunk_rows);

/* Components only (compute_pc, sif_functions.py:58-67, on the SIF embedding): ids H2D || embed of a chunk -> its
 * Gram added to the running sum in chunk order -> one solve.  Device memory is two id chunks + one embedding chunk
 * + the Gram / solve scratch (+ the pre-scaled table for large batches), whatever N is.  N < d runs as one chunk
 * (the start block X^T Omega needs every row).  Omega_host as for mmb_sif_embedding_host; pc_host: npc x d
 * float32, npc in [1, 22]; d <= 512; N >= 1.  The kernel variant is decided on the whole N, so pc_host equals
 * mmb_sif_embedding_host's at the same chunk_rows wherever each chunk of that call runs the whole batch's variant:
 * it decides the CTA-per-utterance rule (L >= 256, N < 16 SMs) per chunk, so a short last chunk of long
 * utterances may run another kernel there.  With chunk_rows >= N it equals mmb_sif_embedding's pc.  Synchronous. */
MMB_API int mmb_sif_fit_host(const float* table_dev, int64_t V, int d, const float* vocab_w_dev,
                             const int64_t* x_host, int64_t N, int64_t L, int npc, const double* Omega_host,
                             float* pc_host, int gram_mode, int64_t chunk_rows);

/* The *_host entry points take their staging buffers from a private stream-ordered pool per device
 * that keeps freed blocks for the next call; this returns all but `keep_bytes` of them to the driver. */
MMB_API int mmb_host_pipeline_trim(size_t keep_bytes);

/* ---------------------------------------------------------------- multi-GPU (SURVEY 8e) */
/* The reference has no distributed code; utterances shard over the GPUs of one box and the only
 * exchange is the sum of the per-rank Grams (and, for N < d, of the start blocks).  These entry
 * points do that sum over NVLink peer memory inside the kernel that finishes the Gram, one
 * process per GPU:
 *   every rank allocates one exchange buffer (mmb_comm_alloc), exports its 64-byte CUDA IPC
 *   handle (mmb_comm_export), the host side all-gathers the handles (torch.distributed), and
 *   opens the peers' buffers (mmb_comm_open).  `bufs` is a HOST array of `world` device
 *   pointers in rank order (bufs[rank] = the rank's own buffer); `epoch` is a counter > 0 that
 *   every rank advances by one per call (same call sequence on all ranks); world <= 8.
 * Sums are taken in rank order, so all ranks obtain identical bits.  A peer that never arrives
 * sets MMB_STATUS_COMM_TIMEOUT in `status` after ~4 s instead of hanging.                    */
MMB_API size_t mmb_comm_bytes(void);
/* Capacity of one exchange slot: the largest vector mmb_allreduce_peer sums in one call (4 MiB). */
MMB_API size_t mmb_comm_slot_bytes(void);
MMB_API int mmb_comm_alloc(void** buf);
MMB_API int mmb_comm_free(void* buf);
MMB_API int mmb_comm_export(void* buf, void* handle64);
MMB_API int mmb_comm_open(const void* handle64, void** peer_buf);
MMB_API int mmb_comm_close(void* peer_buf);
/* x (n elements, float32 or float64 when is_f64 != 0; n * elem size <= 4 MiB) <- sum over ranks,
 * in rank order (identical bits everywhere).  Besides the Gram this carries the flat head-parameter
 * gradient of the data-parallel MMB step (843,400 floats, SURVEY 8e "MMB training") and the
 * cross-rank BatchNorm statistics.  Cooperative launch, grid-stride.                          */
MMB_API int mmb_allreduce_peer(void* x, int64_t n, int is_f64, int rank, int world, void* const* bufs,
                               uint64_t epoch, int* status, mmb_stream_t stream);
/* A rank that cannot take part in the exchange of `epoch` (it failed before its mmb_*_peer call)
 * tells its peers so: their wait ends at once with MMB_STATUS_COMM_TIMEOUT instead of after ~4 s.
 * The communicator is unusable afterwards.                                                     */
MMB_API int mmb_comm_abort(int rank, int world, void* const* bufs, uint64_t epoch, mmb_stream_t stream);
/* mmb_gram followed by the all-reduce of G: on the tcgen05 path the cross-CTA reduction of the
 * Gram partials and the cross-rank exchange are ONE kernel.  N may be 0 on a rank.           */
MMB_API int mmb_gram_allreduce_peer(const float* X, int64_t N, int d, float* G, void* ws, size_t ws_bytes,
                                    int mode, int rank, int world, void* const* bufs, uint64_t epoch,
                                    int* status, mmb_stream_t stream);

/* mmb_sif_embedding_host for one rank's block of a split of N_global utterances (N_global >= d):
 * the same chunked H2D / embed / Gram pipeline, then the sum of the ranks' Grams over NVLink peer
 * memory (mmb_allreduce_peer on the running sum), the replicated solve and the projection
 * overlapped with the D2H.  All ranks call it with the same epoch; N_local may be 0.           */
MMB_API int mmb_sif_embedding_host_peer(const float* table_dev, int64_t V, int d, const float* vocab_w_dev,
                                const int64_t* x_host, int64_t N_local, int64_t L, int npc,
                                const double* Omega_host, void* emb_host, int emb_f64, float* pc_host,
                                int gram_mode, int64_t chunk_rows, int64_t N_global, int rank, int world,
                                void* const* bufs, uint64_t epoch);

/* ---------------------------------------------------------------- MMB (A6-A9) ----- */
/* In this section the pointer tables (W, b, out, seg_val ...) are HOST arrays of DEVICE
 * pointers; the library copies them into kernel parameters (<= 16 heads, <= 8 modalities of
 * <= 4 segments each).                                                                  */

/* AudioVisualGeneratorMultimodal.forward -- models.py:187-202, all heads in one launch.
 * z (B, d) is the (already normalised) latent batch.  Head h has weight W[h] (D[h], d) and
 * bias b[h] (D[h]) (nn.Linear layout); is_log_sigma[h] != 0 selects the exp() epilogue
 * (sigma = exp(.), models.py:199).  out[h] is (B, D[h]).                                */
MMB_API int mmb_heads_forward(const float* z, int B, int d, int n_heads, const float* const* W,
                      const float* const* b, const int* D, const int* is_log_sigma,
                      float* const* out, mmb_stream_t stream);
/* Backward of the above given gout[h] (B, D[h]) = d loss / d pre-activation of head h:
 * dz (B, d) = sum_h gout[h] W[h];  dW[h] (D[h], d) = gout[h]^T z;  db[h] (D[h]) = column sums.
 * dz, dW, db may be NULL (frozen heads, reference models.py:173-178).  dz is a split-K product
 * (sum of D[h] in the thousands spread over ~100 CTAs, partials added in a fixed order): `ws`
 * must hold mmb_heads_backward_workspace_bytes(B, d, n_heads, D) bytes when dz != NULL.   */
MMB_API size_t mmb_heads_backward_workspace_bytes(int B, int d, int n_heads, const int* D);
MMB_API int mmb_heads_backward(const float* z, int B, int d, int n_heads, const float* const* W,
                       const int* D, const float* const* gout, float* dz, float* const* dW,
                       float* const* db, void* ws, size_t ws_bytes, mmb_stream_t stream);

/* get_log_prob_matrix's combination -- losses.py:267-272: out[b] = other_w * sum_m lp[m][b] + word_w * wlp[b]
 * (lp is (M, B) row-major) and its backward, one launch each instead of torch's sum / mul / mul / add chain.
 * When other_w_dev / word_w_dev are non-NULL the weights are read from those device scalars instead.   */
MMB_API int mmb_combine_lp(const float* lp, const float* wlp, int M, int B, float other_w, float word_w,
                           const float* other_w_dev, const float* word_w_dev, float* out, mmb_stream_t stream);
MMB_API int mmb_combine_lp_backward(const float* g, int M, int B, float other_w, float word_w,
                                    const float* other_w_dev, const float* word_w_dev, float* g_lp, float* g_wlp,
                                    mmb_stream_t stream);
/* Launch-count helpers of the step (B = 64: every torch element-wise op is a launch).
 * mmb_scale_multi: out[i] (B, D[i]) = in[i] * row[i][b] * elem[i][b][f] for n <= 16 tensors in one
 * launch (row / elem tables or entries may be NULL = 1): the chain rule through the per-modality
 * log-likelihoods (12 multiplies per MMB2 step) and d sigma / d log_sigma = sigma (6 more).
 * mmb_gather_multi: dst[i] (B, W[i]) = src[i][idx[b]] for n <= 16 row-major tensors sharing one
 * int64 index vector: the batch tuple of MMData.__getitem__ (utils.py:231-233) in one launch.   */
MMB_API int mmb_scale_multi(int n, int B, const int* D, const float* const* in, const float* const* row,
                    const float* const* elem, float* const* out, mmb_stream_t stream);
MMB_API int mmb_gather_multi(int n, int B, const int64_t* idx, const float* const* src, const int64_t* W,
                     float* const* dst, mmb_stream_t stream);

/* get_normal_log_prob -- losses.py:13-34 for n_mod modalities in ONE launch: value and the
 * analytic gradients (SURVEY.md Appendix A.4).  Modality m is the concatenation along the
 * feature axis (the torch.cat of simplesif.py:94-113, never materialised) of n_seg[m]
 * segments; segments are listed modality after modality in seg_val / seg_mask / seg_F:
 *   seg_val[s], seg_mask[s]: (B, T, seg_F[s]) values and float mask;
 *   mu[m], sigma[m]: (B, D_m), D_m = sum of the modality's seg_F;
 *   lp: (n_mod, B) = sum_{t,f} mask * (log(1/sqrt(2 pi sigma^2)) - (x-mu)^2 / (2 sigma^2));
 *   dmu[m], dsigma[m]: (B, D_m) = d lp[m] / d mu, d sigma (tables or entries may be NULL).
 * `status` gets MMB_STATUS_NONFINITE if any lp is not finite (losses.py:258-264).        */
MMB_API int mmb_gauss_ll(int B, int T, int n_mod, const int* n_seg, const float* const* seg_val,
                 const float* const* seg_mask, const int* seg_F, const float* const* mu,
                 const float* const* sigma, float* lp, float* const* dmu, float* const* dsigma,
                 int* status, mmb_stream_t stream);

/* The same likelihood from per-utterance moments.  An utterance's data does not change between
 * optimisation steps (only mu and sigma do), so the sums over time are taken ONCE per dataset:
 *   mmb_gauss_moments: val, mask (N, T, F) -> stats (N, 3, F) = [S0 = sum_t m | mean = sum_t m x / S0 |
 *   M2 = sum_t m (x - mean)^2] (S0 = 0 gives mean = M2 = 0);
 *   mmb_gauss_ll_stats: mmb_gauss_ll with seg_stats[s] = the (B, 3, seg_F[s]) moments of the batch rows in
 *   place of seg_val / seg_mask, using  sum_t m (x - mu)^2 = M2 + S0 (mean - mu)^2  (exact, cancellation-free):
 *   3 floats per (utterance, feature) per step instead of 2 T.                                            */
MMB_API int mmb_gauss_moments(const float* val, const float* mask, int64_t N, int T, int F, float* stats,
                      mmb_stream_t stream);
MMB_API int mmb_gauss_ll_stats(int B, int n_mod, const int* n_seg, const float* const* seg_stats, const int* seg_F,
                       const float* const* mu, const float* const* sigma, float* lp, float* const* dmu,
                       float* const* dsigma, int* status, mmb_stream_t stream);

/* get_word_log_prob_angular2 -- losses.py:68-95, value + d/d latents (Appendix A.5).
 *   latents (B, d); table (V, d) and inv_norm (V) = 1/max(||row||, 1e-8) from
 *   mmb_row_inv_norm (torch CosineSimilarity's clamp); sent: token vectors, element
 *   (b, t, k) at sent[b*sent_stride_b + t*sent_stride_t + k]; word_w (B, L) dense; tmask
 *   element (b, t) at tmask[b*tmask_stride_b + t*tmask_stride_t] (= mask[:, :, 0]);
 *   a = 1e-3 (simplesif.py:513).  lp (B); grad (B, d) = d lp / d latents.
 *   The partition term is a (B, d) x (d, V) product with an acos epilogue and its gradient a
 *   (B, V) x (V, d) product -- no (B, V, d) broadcast temporaries.
 *   ws >= mmb_word_ll_workspace_bytes(B, V, d).                                          */
MMB_API int mmb_row_inv_norm(const float* X, int64_t n, int d, float* inv_norm, mmb_stream_t stream);
MMB_API size_t mmb_word_ll_workspace_bytes(int B, int64_t V, int d);
MMB_API int mmb_word_ll(const float* latents, int B, int d, const float* table, const float* inv_norm,
                int64_t V, const float* sent, int64_t sent_stride_b, int64_t sent_stride_t,
                const float* word_w, const float* tmask, int64_t tmask_stride_b,
                int64_t tmask_stride_t, int L, float a, float* lp, float* grad, void* ws,
                size_t ws_bytes, int* status, mmb_stream_t stream);

/* The same term when the token vectors are rows of `table` (reference simplesif.py:319-340 builds
 * text = word_embeddings[ids]; SURVEY.md 8f N3): ids (B, L) int64, row b at ids + b*ids_stride_b, replace
 * `sent`.  The token cosines are read out of the (B, V) cosine matrix of the partition term and the token
 * gradient rides its (B, V) x (V, d) product, so no (B, L, d) tensor is read: the cost is independent of
 * L*d.  tmask may be NULL (= ids != 0).  Ids outside [0, V) set MMB_STATUS_BAD_INDEX.  Needs
 * (V + L) * 4 bytes of shared memory per utterance (<= 200 KiB), else MMB_E_UNSUPPORTED.
 *   ws >= mmb_word_ll_ids_workspace_bytes(B, V, d).                                                    */
MMB_API size_t mmb_word_ll_ids_workspace_bytes(int B, int64_t V, int d);
MMB_API int mmb_word_ll_ids(const float* latents, int B, int d, const float* table, const float* inv_norm,
                    int64_t V, const int64_t* ids, int64_t ids_stride_b, const float* word_w,
                    const float* tmask, int64_t tmask_stride_b, int64_t tmask_stride_t, int L, float a,
                    float* lp, float* grad, void* ws, size_t ws_bytes, int* status, mmb_stream_t stream);

/* ---------------------------------------------------------------- closed form (N1) */
/* estimate_embedding_overall_gpu2 -- sif2.py:164-208 with calc_weights sif2.py:103-114 (call site
 * simplesif.py:808-880): gradient-free latents as the weight-normalised, L2-normalised sum of the
 * SIF text average and per-modality q_mean W_mu + q_sigma W_log_sigma terms.
 * Step 1, one pass over the base tensors (modalities = concatenations of segments, as in
 * mmb_gauss_ll): S1[m], S2[m] (N, D_m) = sums over time of q_mean, q_sigma, and
 * tw_part (n_mod, N) = their sums over features.  Step 2: prod (N, d) = sum_m S1[m] W_mu[m] +
 * S2[m] W_ls[m] with mmb_heads_backward (dz only; gout = S1/S2, W = the (D_m, d) weights).
 * Step 3: out (N, d) = normalise((sum_t sent_w[n,t] emb[n,t,:] + prod) / tw).              */
MMB_API int mmb_closed_form_stats(int N, int T, int n_mod, const int* n_seg, const float* const* seg_val,
                          const int* seg_F, const float* const* b_mu, const float* const* b_ls,
                          float* const* S1, float* const* S2, float* tw_part, mmb_stream_t stream);
MMB_API int mmb_closed_form_finish(int N, int L, int d, const float* sent_w, const float* emb,
                           const float* prod, const float* tw_part, int n_mod, float* out,
                           mmb_stream_t stream);

/* ---------------------------------------------------------------- preprocessing (N3) */
/* normalize_data utils.py:155-191 + add_positional_embeddings utils.py:130-153 + the mask
 * extension of simplesif.py:369-375 on the device, for one feature tensor x (N, T, F_in) float32.
 * mmb_feature_minmax: per-column min / max over all N*T rows (the split's own statistics).
 * mmb_prep_features: keep[] (device, F_out ints, ascending) lists the non-constant source columns
 * (max > min; the reference drops constant AUDIO features only -- pass all columns for the visual
 * tensor); out / mask are (N, T, F_out + pos_embed_dim): value (x + min) * 2 / (max - min) - 1
 * (the reference adds the minimum), exact zeros -> -10 with mask 0, then pos_embed_dim position
 * columns with the reference's first-axis quirk and mask 1.                                 */
/* update_masks simplesif.py:36-40: mask[i] = ids[i] != 0 as float (the (N, L, d) broadcast is a stride-0
 * view on the caller's side); update_masks_vect simplesif.py:42-47: mask[r] = all(x[r, :] != 0) for the
 * (N*T, F) rows of an aligned text tensor.                                                         */
MMB_API int mmb_token_mask(const int64_t* ids, int64_t n, float* mask, mmb_stream_t stream);
MMB_API int mmb_step_mask(const float* x, int64_t rows, int F, float* mask, mmb_stream_t stream);
MMB_API size_t mmb_feature_minmax_workspace_bytes(int64_t rows, int F);
MMB_API int mmb_feature_minmax(const float* x, int64_t rows, int F, float* mn, float* mx, void* ws,
                       size_t ws_bytes, mmb_stream_t stream);
MMB_API int mmb_prep_features(const float* x, int64_t N, int T, int F_in, const int* keep, int F_out,
                      int pos_embed_dim, const float* mn, const float* mx, float* out, float* mask,
                      mmb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MMB_B200_H */
