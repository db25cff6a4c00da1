// Principal components from the Gram (reference: sif_functions.py:58-67 compute_pc, i.e.
// scikit-learn TruncatedSVD(n_components=npc, n_iter=7, random_state=0) -> randomized SVD).
//
// sklearn's output is a function of G = X^T X and the seeded start block only (SURVEY.md
// section 7 H1; oracle/sif_oracle.py:compute_pc_from_gram):
//   Q = orth(S0); repeat n_iter: Q = orth(G Q);  Y = G Q;  T = Q^T Y
//   N >= d : components = top eigenvectors of Y T^-1 Y^T = left singular vectors of
//            W = Y R^-1 with T = R^T R            (sklearn: right singular vectors of Q_x^T X)
//   N <  d : components = Q * top eigenvectors of T   (sklearn works on X^T: Rayleigh-Ritz)
//   rows unit-normalised, largest-|entry| of each row made positive (svd_flip, v-based).
// The problem is d x k (d <= 512, k = npc + 10 <= 32).  It runs in FP64 entirely on the device:
// no host round trip between the Gram and the projection pass (SURVEY.md H5).  orth() is
// CholeskyQR with rank-deficient columns dropped, repeated (CholeskyQR2) where the result must be
// orthonormal and not only span the right space.
//
// The chain of 2 n_iter + 4 dependent steps is what every rank waits for between the Gram
// all-reduce and the projection pass, so it is organised for latency (run by one CTA, the chain is
// instruction-issue bound and took 1.35 ms on a B200).  It runs as n_iter + 3 small kernels on one
// stream:
//   prep   : S0 -> column-major Y_0, per-CTA partials of Y_0^T Y_0;
//   iter i : EVERY CTA sums the partials (fixed order), factorises the k x k matrix and forms
//            Q_i = orth(Y_i) for all d rows redundantly -- no CTA ever waits for a serial CTA --
//            then computes ITS 8 rows of Y_{i+1} = G Q_i (FP64, G rows staged in shared memory,
//            j split over thread groups and summed in fixed order) and the partials of
//            Y_{i+1}^T Y_{i+1} (last iteration: of T = Q^T Y, plus its rows of Q);
//   final  : one CTA: Rayleigh-Ritz on the k x k problem (Cholesky + parallel-ordered Jacobi on
//            several warps), components, unit norm, sklearn's sign rule.
// Kernel boundaries are the grid-wide barriers.  Everything is summed in a fixed order, so the
// result is deterministic and identical on every rank.
#include "common.cuh"

namespace mmb {

constexpr int kPcMaxK = 32;
constexpr int kPcmRows = 8;        // rows of Y per CTA in the iteration kernels
constexpr int kPcmThreads = 320;

struct PcmSmall {
  double S[kPcMaxK + 1][kPcMaxK + 1];
  double Vv[kPcMaxK][kPcMaxK + 1];
  double P[kPcMaxK][kPcMaxK + 1];   // scratch of pcm_top1
  double lam[kPcMaxK];
  double rc[kPcMaxK / 2], rs[kPcMaxK / 2];
  double red[8];
  int rp[kPcMaxK / 2], rq[kPcMaxK / 2];
  int drop[kPcMaxK];
  int order[kPcMaxK];
  int flag;
};

// 1/sqrt(x), 1/x: hardware FP32 seed + two Newton steps in FP64 (full double precision for
// normal-range arguments; far fewer instructions than the IEEE-exact library sequences, which
// matters because these phases are issue-bound on a single warp).
__device__ __forceinline__ double pcm_rsqrt(double x) {
  if (!(x > 1e-30 && x < 1e30)) return rsqrt(x);
  double r = (double)rsqrtf((float)x);
  r = r * fma(-0.5 * x, r * r, 1.5);
  return r * fma(-0.5 * x, r * r, 1.5);
}
__device__ __forceinline__ double pcm_rcp(double x) {
  const double ax = fabs(x);
  if (!(ax > 1e-30 && ax < 1e30)) return 1.0 / x;
  double r = (double)__frcp_rn((float)x);
  r = r * fma(-x, r, 2.0);
  return r * fma(-x, r, 2.0);
}

// Upper Cholesky S = R^T R in place by warp 0, left-looking: for column step c lane j >= c forms
// v_j = S[c][j] - sum_{a<c} R[a][c] R[a][j] AND the pivot v_c itself (redundantly, so that no
// value has to cross lanes inside the k-step serial chain), then scales by 1/sqrt(v_c).
// 1/sqrt comes from the FP32 hardware seed on the pivot scaled into (0, 1] plus `newton`
// Newton steps in FP64 (1: ~5e-15 relative, enough where only the span of Q matters; 2: full
// double precision).  Columns whose pivot is not positive relative to the largest diagonal
// entry are dropped (they lie in the span of earlier columns): row c of R becomes 0 and
// lam[c] = 1/R[c][c] = 0.  Ends with __syncthreads().
__device__ __forceinline__ void pcm_cholesky(PcmSmall& sm, int k, int newton) {
  if (threadIdx.x < 32) {
    const int j = threadIdx.x;
    double dmax = (j < k) ? sm.S[j][j] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
    const bool usable = dmax > 0.0 && dmax < 1e300;
    const double rs_dmax = usable ? rsqrt(dmax) : 0.0;   // once per factorisation
    const double inv_dmax = rs_dmax * rs_dmax;
    for (int c = 0; c < k; ++c) {
      double vj = 0.0, vc = 0.0;
      if (j >= c && j < k) {
        vj = sm.S[c][j];
        vc = sm.S[c][c];
        for (int a = 0; a < c; ++a) {
          const double rac = sm.S[a][c];
          vj = fma(-rac, sm.S[a][j], vj);
          vc = fma(-rac, rac, vc);
        }
        const double x = vc * inv_dmax;                  // in (1e-26, ~1]: safe for the FP32 seed
        const bool bad = !(x > 1e-26) || !(x < 1e30);
        double r = (double)rsqrtf((float)x);
        r = r * fma(-0.5 * x, r * r, 1.5);
        if (newton > 1) r = r * fma(-0.5 * x, r * r, 1.5);
        const double rinv = bad ? 0.0 : r * rs_dmax;
        if (j == c) {
          sm.drop[c] = bad;
          sm.S[c][c] = bad ? 1.0 : vc * rinv;   // sqrt(pivot)
          sm.lam[c] = rinv;
        } else {
          sm.S[c][j] = vj * rinv;
        }
      }
      __syncwarp();
    }
  }
  __syncthreads();
}

// row <- row * R^-1, right-looking (after q[c] is final, every later column is updated at
// once: the dependent chain is k multiply-adds, not k^2 / 2).
template <int KMAX>
__device__ __forceinline__ void pcm_solve_row(const PcmSmall& sm, double (&q)[KMAX], int k) {
#pragma unroll
  for (int c = 0; c < KMAX; ++c) {
    if (c < k) {
      q[c] *= sm.lam[c];
#pragma unroll
      for (int b = c + 1; b < KMAX; ++b)
        if (b < k) q[b] = fma(-q[c], sm.S[c][b], q[b]);
    }
  }
}

// S[a][b] = sum_i A[a][i] B[b][i] over all d rows (A, B column-major [KP][DP] in shared memory);
// one (a, b) pair per group of 4 threads (row quarters, combined in fixed order by shuffles).
__device__ __forceinline__ void pcm_small_gram(PcmSmall& sm, const double* A, const double* B, int d, int k,
                                               int DP, bool symmetric) {
  const int sub = threadIdx.x & 3, grp = threadIdx.x >> 2, ngrp = kPcmThreads >> 2;
  const int npairs = k * k;
  for (int p0 = 0; p0 < npairs; p0 += ngrp) {
    const int p = p0 + grp;
    const int a = p < npairs ? p / k : 0, b = p < npairs ? p - (p / k) * k : 0;
    double s0 = 0.0, s1 = 0.0;
    if (p < npairs && !(symmetric && b < a)) {
      const double* pa = A + (size_t)a * DP;
      const double* pb = B + (size_t)b * DP;
      int i = sub;
      for (; i + 4 < d; i += 8) {
        s0 = fma(pa[i], pb[i], s0);
        s1 = fma(pa[i + 4], pb[i + 4], s1);
      }
      if (i < d) s0 = fma(pa[i], pb[i], s0);
    }
    double sacc = s0 + s1;
    sacc += __shfl_xor_sync(0xffffffffu, sacc, 1);
    sacc += __shfl_xor_sync(0xffffffffu, sacc, 2);
    if (sub == 0 && p < npairs && !(symmetric && b < a)) {
      sm.S[a][b] = sacc;
      if (symmetric) sm.S[b][a] = sacc;
    }
  }
  __syncthreads();
}

// sum_c part[c * stride] over the nbp partial slots (nbp = CTA count rounded up to 8, <= 64; the
// pad slots hold zeros) in CTA order.  All loads are issued before the first add, so the sum
// costs one L2 round trip instead of one per unrolled batch.
__device__ __forceinline__ double pcm_sum_partials(const double* __restrict__ part, size_t stride, int nbp) {
  double v[8][8];
#pragma unroll
  for (int ch = 0; ch < 8; ++ch) {
    if (ch * 8 < nbp) {
#pragma unroll
      for (int u = 0; u < 8; ++u) v[ch][u] = part[(size_t)(ch * 8 + u) * stride];
    }
  }
  double s = 0.0;
#pragma unroll
  for (int ch = 0; ch < 8; ++ch) {
    if (ch * 8 < nbp) {
#pragma unroll
      for (int u = 0; u < 8; ++u) s += v[ch][u];
    }
  }
  return s;
}

__global__ void __launch_bounds__(128)
    pcm_prep_kernel(const double* __restrict__ S0, int d, int k, int KP, int DP, double* __restrict__ Y0,
                    double* __restrict__ Spart, double* __restrict__ SpartB, int nbp) {
  __shared__ double ys[kPcmRows][kPcMaxK];
  const int row0 = blockIdx.x * kPcmRows;
  if (blockIdx.x == 0) {   // zero the pad slots [gridDim.x, nbp) of both partial buffers
    const int n = (nbp - (int)gridDim.x) * KP * KP;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      Spart[(size_t)gridDim.x * KP * KP + i] = 0.0;
      SpartB[(size_t)gridDim.x * KP * KP + i] = 0.0;
    }
  }
  for (int i = threadIdx.x; i < kPcmRows * KP; i += blockDim.x) {
    const int r = i / KP, c = i - r * KP, row = row0 + r;
    const double v = (row < d && c < k) ? S0[(size_t)row * k + c] : 0.0;
    ys[r][c] = v;
    if (row < d) Y0[(size_t)c * DP + row] = v;
  }
  __syncthreads();
  for (int p = threadIdx.x; p < k * k; p += blockDim.x) {
    const int a = p / k, b = p - a * k;
    double s = 0.0;
#pragma unroll
    for (int r = 0; r < kPcmRows; ++r) s = fma(ys[r][a], ys[r][b], s);
    Spart[(size_t)blockIdx.x * KP * KP + a * KP + b] = s;
  }
}

template <int KMAX>
__global__ void __launch_bounds__(kPcmThreads)
    pcm_iter_kernel(const float* __restrict__ G, int d, int k, int KP, int DP, int nb,
                    const double* __restrict__ Yprev, double* __restrict__ Ynext, double* __restrict__ Qout,
                    const double* __restrict__ SpartIn, double* __restrict__ SpartOut, int passes, int last) {
  extern __shared__ __align__(16) unsigned char pcm_smem[];
  PcmSmall& sm = *reinterpret_cast<PcmSmall*>(pcm_smem);
  double* Qt = reinterpret_cast<double*>(pcm_smem + ((sizeof(PcmSmall) + 15) & ~(size_t)15));   // [KP][DP]
  double* red = Qt + (size_t)KP * DP;                                // [JS][kPcmRows][KP]
  const int ng = KP / 4;                                             // 4-column groups
  const int items = kPcmRows * ng;                                   // (row, column group) tiles
  const int JS = kPcmThreads / items;                                // j slices
  double* ys = red + (size_t)JS * kPcmRows * KP;                     // [kPcmRows][KP]
  float* Gs = reinterpret_cast<float*>(ys + kPcmRows * KP);          // [kPcmRows][d]
  const int row0 = blockIdx.x * kPcmRows;

  // Programmatic dependent launch: let the next kernel of the chain start its own prologue now,
  // stage this CTA's G rows (independent of the previous kernel), and only then wait for the
  // previous kernel's Y / partials to be complete and visible.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  for (int i = threadIdx.x; i < kPcmRows * d; i += kPcmThreads) {
    const int r = i / d, row = row0 + r;
    Gs[i] = row < d ? __ldg(G + (size_t)row * d + (i - r * d)) : 0.f;
  }
  asm volatile("griddepcontrol.wait;" ::: "memory");
  // S = sum of the per-CTA partials, CTA order
  for (int p = threadIdx.x; p < k * k; p += kPcmThreads) {
    const int a = p / k, b = p - a * k;
    sm.S[a][b] = pcm_sum_partials(SpartIn + a * KP + b, (size_t)KP * KP, (nb + 7) & ~7);
  }
  // this thread's row of Y (loaded before the factorisation so that its latency hides behind it)
  const int myrow = threadIdx.x;
  double q[KMAX];
#pragma unroll
  for (int c = 0; c < KMAX; ++c) q[c] = (c < k && myrow < d) ? Yprev[(size_t)c * DP + myrow] : 0.0;
  __syncthreads();
  pcm_cholesky(sm, k, last ? 2 : 1);
  // Q = Y R^-1 for all rows (redundantly in every CTA), column-major in shared memory
  if (myrow < DP) {
    pcm_solve_row<KMAX>(sm, q, k);
#pragma unroll
    for (int c = 0; c < KMAX; ++c)
      if (c < KP) Qt[(size_t)c * DP + myrow] = q[c];
  }
  for (int row = myrow + kPcmThreads; row < DP; row += kPcmThreads) {   // d > 320 only
    double q2[KMAX];
#pragma unroll
    for (int c = 0; c < KMAX; ++c) q2[c] = (c < k && row < d) ? Yprev[(size_t)c * DP + row] : 0.0;
    pcm_solve_row<KMAX>(sm, q2, k);
#pragma unroll
    for (int c = 0; c < KMAX; ++c)
      if (c < KP) Qt[(size_t)c * DP + row] = q2[c];
  }
  __syncthreads();
  for (int pass = 1; pass < passes; ++pass) {   // CholeskyQR2
    pcm_small_gram(sm, Qt, Qt, d, k, DP, true);
    pcm_cholesky(sm, k, 2);
    for (int row = threadIdx.x; row < d; row += kPcmThreads) {
      double q[KMAX];
#pragma unroll
      for (int c = 0; c < KMAX; ++c) q[c] = c < k ? Qt[(size_t)c * DP + row] : 0.0;
      pcm_solve_row<KMAX>(sm, q, k);
#pragma unroll
      for (int c = 0; c < KMAX; ++c)
        if (c < k) Qt[(size_t)c * DP + row] = q[c];
    }
    __syncthreads();
  }
  // Y rows of this CTA: tile = (row, 4 columns), j split over JS thread groups
  {
    const int t = threadIdx.x;
    const int js = t / items, it = t - js * items;
    if (js < JS) {
      const int r = it / ng, c0 = (it - r * ng) * 4;
      const int jlen = (d + JS - 1) / JS;
      const int j0 = js * jlen, j1 = (j0 + jlen) < d ? (j0 + jlen) : d;
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
      const float* g = Gs + (size_t)r * d;
      const double* q0 = Qt + (size_t)c0 * DP;
#pragma unroll 4
      for (int j = j0; j < j1; ++j) {
        const double gv = (double)g[j];
        a0 = fma(gv, q0[j], a0);
        a1 = fma(gv, q0[DP + j], a1);
        a2 = fma(gv, q0[2 * DP + j], a2);
        a3 = fma(gv, q0[3 * DP + j], a3);
      }
      double* o = red + ((size_t)js * kPcmRows + r) * KP + c0;
      o[0] = a0; o[1] = a1; o[2] = a2; o[3] = a3;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kPcmRows * KP; i += kPcmThreads) {
    const int r = i / KP, c = i - r * KP, row = row0 + r;
    double s = 0.0;
    for (int js = 0; js < JS; ++js) s += red[((size_t)js * kPcmRows + r) * KP + c];
    if (c >= k || row >= d) s = 0.0;
    ys[i] = s;
    if (row < d) {
      Ynext[(size_t)c * DP + row] = s;
      if (last) Qout[(size_t)c * DP + row] = Qt[(size_t)c * DP + row];
    }
  }
  __syncthreads();
  // partials for the next kernel: Y^T Y of these rows, or (last) T = Q^T Y
  for (int p = threadIdx.x; p < k * k; p += kPcmThreads) {
    const int a = p / k, b = p - a * k;
    double s = 0.0;
#pragma unroll
    for (int r = 0; r < kPcmRows; ++r) {
      const int row = row0 + r;
      const double left = last ? (row < d ? Qt[(size_t)a * DP + row] : 0.0) : ys[r * KP + a];
      s = fma(left, ys[r * KP + b], s);
    }
    SpartOut[(size_t)blockIdx.x * KP * KP + a * KP + b] = s;
  }
}

// Symmetric eigenproblem of sm.S (k <= 32), all warps of the CTA: Jacobi with the round-robin
// ("chess tournament") ordering: per round k/2 disjoint rotations; the two-sided update
// S <- J^T S J is applied 2x2 block by 2x2 block (one thread per block) while other threads
// rotate the eigenvector columns; rotation parameters by the first k/2 threads.
__device__ __forceinline__ void pcm_jacobi(PcmSmall& sm, int k) {
  const int t = threadIdx.x;
  const int m = (k + 1) & ~1, half = m >> 1;
  for (int i = t; i < kPcMaxK * (kPcMaxK + 1); i += kPcmThreads) {
    const int r = i / (kPcMaxK + 1), c = i - r * (kPcMaxK + 1);
    if (r < kPcMaxK) sm.Vv[r][c] = (r == c) ? 1.0 : 0.0;
  }
  if (t <= m) { sm.S[t][k] = 0.0; sm.S[k][t] = 0.0; }   // dummy index of an odd k: never rotated
  __syncthreads();
  for (int sweep = 0; sweep < 30 && m > 1; ++sweep) {
    if (t < 32) {
      double off = 0.0, dg = 0.0;
      if (t < k) {
        for (int c = 0; c < k; ++c) {
          const double v = sm.S[t][c];
          if (c > t) off = fma(v, v, off);
          if (c == t) dg = v * v;
        }
      }
      off = warp_sum(off);
      dg = warp_sum(dg);
      if (t == 0) sm.flag = !(off > 1e-27 * dg);   // off-diagonal mass below ~3e-14 of the diagonal
    }
    __syncthreads();
    if (sm.flag) break;
    for (int r = 0; r < m - 1; ++r) {
      if (t < half) {
        int p, q;
        if (t == 0) { p = m - 1; q = r; }
        else { p = r + t; if (p >= m - 1) p -= m - 1; q = r - t; if (q < 0) q += m - 1; }
        if (p > q) { const int x = p; p = q; q = x; }
        double c = 1.0, s = 0.0;
        if (q < k) {
          const double apq = sm.S[p][q], app = sm.S[p][p], aqq = sm.S[q][q];
          if (fabs(apq) > 1e-300 && apq * apq > 1e-34 * fabs(app * aqq)) {
            // t = sgn(theta) / (|theta| + sqrt(theta^2 + 1)), theta = (aqq - app) / (2 apq)
            const double dl = aqq - app, tw = 2.0 * apq;
            const double h2 = fma(dl, dl, tw * tw);
            const double h = h2 * pcm_rsqrt(h2);
            const double tt = (dl >= 0.0 ? tw : -tw) * pcm_rcp(fabs(dl) + h);
            c = pcm_rsqrt(fma(tt, tt, 1.0));
            s = tt * c;
          }
        }
        sm.rp[t] = p; sm.rq[t] = q; sm.rc[t] = c; sm.rs[t] = s;
      }
      __syncthreads();
      if (t < half * half) {            // 2x2 block (e1, e2): B <- J1^T B J2
        const int e1 = t / half, e2 = t - e1 * half;
        const int p1 = sm.rp[e1], q1 = sm.rq[e1], p2 = sm.rp[e2], q2 = sm.rq[e2];
        const double c1 = sm.rc[e1], s1 = sm.rs[e1], c2 = sm.rc[e2], s2 = sm.rs[e2];
        const double b00 = sm.S[p1][p2], b01 = sm.S[p1][q2], b10 = sm.S[q1][p2], b11 = sm.S[q1][q2];
        // columns (J2): [x0 x1] = [b.0 b.1] J2
        const double x00 = c2 * b00 - s2 * b01, x01 = s2 * b00 + c2 * b01;
        const double x10 = c2 * b10 - s2 * b11, x11 = s2 * b10 + c2 * b11;
        // rows (J1^T)
        double y00 = c1 * x00 - s1 * x10, y01 = c1 * x01 - s1 * x11;
        double y10 = s1 * x00 + c1 * x10, y11 = s1 * x01 + c1 * x11;
        if (e1 == e2 && s1 != 0.0) { y01 = 0.0; y10 = 0.0; }   // the rotated pair is decoupled exactly
        sm.S[p1][p2] = y00; sm.S[p1][q2] = y01; sm.S[q1][p2] = y10; sm.S[q1][q2] = y11;
      } else {                          // eigenvector columns: V <- V J, item = (rotation, row)
        const int nv = kPcmThreads - half * half;
        for (int it = t - half * half; it < half * k; it += nv) {
          const int e = it / k, i = it - e * k;
          const double c = sm.rc[e], s = sm.rs[e];
          const int p = sm.rp[e], q = sm.rq[e];
          const double vp = sm.Vv[i][p], vq = sm.Vv[i][q];
          sm.Vv[i][p] = c * vp - s * vq;
          sm.Vv[i][q] = s * vp + c * vq;
        }
      }
      __syncthreads();
    }
  }
  if (t < k) sm.lam[t] = sm.S[t][t];
  __syncthreads();
  if (t == 0) {   // descending, stable in index
    unsigned used = 0u;
    for (int r = 0; r < k; ++r) {
      int best = -1;
      for (int c = 0; c < k; ++c)
        if (!((used >> c) & 1u) && (best < 0 || sm.lam[c] > sm.lam[best])) best = c;
      used |= 1u << best;
      sm.order[r] = best;
    }
  }
  __syncthreads();
}

// npc == 1 fast path: the top eigenvector of sm.S (symmetric positive semi-definite, k x k)
// without a full eigen-decomposition.  B = S / tr(S) is squared six times (B^64, renormalised
// by its trace each time), which is numerically rank one whenever lambda_2 / lambda_1 < ~0.55;
// its dominant column is polished by three power steps with S itself and accepted only if
// || S v - lambda v || <= 1e-13 lambda.  Otherwise (no spectral gap) the caller falls back to
// the Jacobi solver, so the result never depends on the gap assumption.  On success
// sm.Vv[:, 0] = v and sm.order[0] = 0.  Returns the acceptance flag (uniform over the CTA).
__device__ __forceinline__ bool pcm_top1(PcmSmall& sm, int k) {
  const int t = threadIdx.x;
  const int i = t / k, j = t - i * k;
  const bool mine = t < k * k;
  double tr = 0.0;
  for (int a = 0; a < k; ++a) tr += sm.S[a][a];
  const bool ok_tr = tr > 0.0 && tr < 1e300;
  double rtr = ok_tr ? pcm_rcp(tr) : 0.0;
  if (mine) sm.Vv[i][j] = sm.S[i][j] * rtr;
  __syncthreads();
  for (int m = 0; m < 6; ++m) {
    double acc = 0.0;
    if (mine)
      for (int l = 0; l < k; ++l) acc = fma(sm.Vv[i][l], sm.Vv[l][j], acc);
    if (mine) sm.P[i][j] = acc;
    __syncthreads();
    double tr2 = 0.0;
    for (int a = 0; a < k; ++a) tr2 += sm.P[a][a];
    rtr = tr2 > 0.0 ? pcm_rcp(tr2) : 0.0;
    if (mine) sm.Vv[i][j] = acc * rtr;
    __syncthreads();
  }
  bool ok = ok_tr;
  if (t < 32) {
    // dominant column = the one with the largest diagonal entry (first on ties)
    double best = -1.0;
    int arg = 0;
    for (int a = 0; a < k; ++a) {
      const double v = sm.Vv[a][a];
      if (v > best) { best = v; arg = a; }
    }
    double v = t < k ? sm.Vv[t][arg] : 0.0;
    double n2 = warp_sum(v * v);
    v *= (n2 > 0.0) ? pcm_rsqrt(n2) : 0.0;
    double lam = 0.0, res = 0.0;
    for (int step = 0; step < 4; ++step) {   // three power steps with S, then the residual
      if (t < k) sm.P[0][t] = v;
      __syncwarp();
      double y = 0.0;
      if (t < k)
        for (int a = 0; a < k; ++a) y = fma(sm.S[t][a], sm.P[0][a], y);
      __syncwarp();
      lam = warp_sum(y * v);
      if (step == 3) {
        const double r = y - lam * v;
        res = warp_sum(r * r);
        break;
      }
      n2 = warp_sum(y * y);
      v = y * ((n2 > 0.0) ? pcm_rsqrt(n2) : 0.0);
    }
    const bool good = ok && lam > 0.0 && res <= 1e-26 * lam * lam;
    if (t < k) sm.P[1][t] = v;
    if (t == 0) sm.flag = good ? 1 : 0;
  }
  __syncthreads();
  ok = sm.flag != 0;
  if (ok) {
    if (t < k) sm.Vv[t][0] = sm.P[1][t];
    if (t == 0) sm.order[0] = 0;
  }
  __syncthreads();
  return ok;
}

template <int KMAX>
__global__ void __launch_bounds__(kPcmThreads)
    pcm_final_kernel(int d, int k, int KP, int DP, int nb, int npc, int transposed,
                     const double* __restrict__ Y, const double* __restrict__ Q,
                     const double* __restrict__ Tpart, float* __restrict__ pc) {
  extern __shared__ __align__(16) unsigned char pcm_smem[];
  PcmSmall& sm = *reinterpret_cast<PcmSmall*>(pcm_smem);
  double* Wt = reinterpret_cast<double*>(pcm_smem + ((sizeof(PcmSmall) + 15) & ~(size_t)15));   // [KP][DP]
  double* cvec = Wt + (size_t)KP * DP;                                                            // [DP]
  asm volatile("griddepcontrol.wait;" ::: "memory");
  for (int p = threadIdx.x; p < k * k; p += kPcmThreads) {
    const int a = p / k, b = p - a * k;
    sm.S[a][b] = pcm_sum_partials(Tpart + a * KP + b, (size_t)KP * KP, (nb + 7) & ~7);
  }
  __syncthreads();
  if (threadIdx.x < k) {   // symmetrise T = Q^T G Q
    const int a = threadIdx.x;
    for (int b = a + 1; b < k; ++b) {
      const double mval = 0.5 * (sm.S[a][b] + sm.S[b][a]);
      sm.S[a][b] = mval;
      sm.S[b][a] = mval;
    }
  }
  __syncthreads();
  if (transposed) {      // Rayleigh-Ritz vectors of G on span(Q)
    for (int i = threadIdx.x; i < KP * DP; i += kPcmThreads) Wt[i] = Q[i];
    __syncthreads();
    if (!(npc == 1 && k * k <= kPcmThreads && pcm_top1(sm, k))) pcm_jacobi(sm, k);
  } else {               // left singular vectors of W = Y R^-1, T = R^T R
    pcm_cholesky(sm, k, 2);
    for (int row = threadIdx.x; row < DP; row += kPcmThreads) {
      double q[KMAX];
#pragma unroll
      for (int c = 0; c < KMAX; ++c) q[c] = (c < k && row < d) ? Y[(size_t)c * DP + row] : 0.0;
      pcm_solve_row<KMAX>(sm, q, k);
#pragma unroll
      for (int c = 0; c < KMAX; ++c)
        if (c < KP) Wt[(size_t)c * DP + row] = q[c];
    }
    __syncthreads();
    pcm_small_gram(sm, Wt, Wt, d, k, DP, true);
    if (!(npc == 1 && k * k <= kPcmThreads && pcm_top1(sm, k))) pcm_jacobi(sm, k);
  }
  for (int c = 0; c < npc; ++c) {
    const int sel = sm.order[c];
    for (int row = threadIdx.x; row < d; row += kPcmThreads) {
      double v = 0.0;
      for (int a = 0; a < k; ++a) v = fma(Wt[(size_t)a * DP + row], sm.Vv[a][sel], v);
      cvec[row] = v;
    }
    __syncthreads();
    if (threadIdx.x < 32) {   // norm + sklearn's sign rule (first arg-max of |v|)
      const int l = threadIdx.x;
      double n2 = 0.0, best = -1.0;
      int arg = 0x7fffffff;
      for (int i = l; i < d; i += 32) {
        const double x = cvec[i];
        n2 = fma(x, x, n2);
        if (fabs(x) > best) { best = fabs(x); arg = i; }
      }
      n2 = warp_sum(n2);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
        if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
      }
      if (l == 0) sm.red[0] = (cvec[arg] < 0.0 ? -1.0 : 1.0) / sqrt(n2);
    }
    __syncthreads();
    for (int row = threadIdx.x; row < d; row += kPcmThreads) pc[(size_t)c * d + row] = (float)(cvec[row] * sm.red[0]);
    __syncthreads();
  }
}

struct PcmPlan {
  int KP, DP, nb, JS;
  size_t blk, spart, smem_iter, smem_final, ws_bytes;
};
static PcmPlan pcm_plan(int d, int k) {
  PcmPlan P;
  P.KP = (k + 3) & ~3;
  P.DP = ((d + 7) & ~7) | 1;   // odd: the 4-column groups of one row land in different banks
  P.nb = (d + kPcmRows - 1) / kPcmRows;
  const int items = kPcmRows * (P.KP / 4);
  P.JS = kPcmThreads / items;
  P.blk = (size_t)P.KP * P.DP;              // doubles per d x k block
  P.spart = (size_t)((P.nb + 7) & ~7) * P.KP * P.KP;     // doubles per partial buffer (padded to 8 slots)
  const size_t small = (sizeof(PcmSmall) + 15) & ~(size_t)15;
  P.smem_iter = small + (P.blk + (size_t)(P.JS > 0 ? P.JS : 1) * kPcmRows * P.KP + kPcmRows * P.KP) * sizeof(double) +
                (size_t)kPcmRows * d * sizeof(float);
  P.smem_final = small + (P.blk + P.DP) * sizeof(double);
  P.ws_bytes = (3 * P.blk + 2 * P.spart) * sizeof(double);
  return P;
}

template <int KMAX>
static int pcm_run(const float* G, int d, const double* S0, int k, int npc, int transposed, int n_iter,
                   float* pc, double* ws, cudaStream_t st) {
  const PcmPlan P = pcm_plan(d, k);
  double* Yb[2] = {ws, ws + P.blk};
  double* Qg = ws + 2 * P.blk;
  double* Sp[2] = {ws + 3 * P.blk, ws + 3 * P.blk + P.spart};
  static bool attr_set = false;
  if (!attr_set) {
    MMB_CUDA(cudaFuncSetAttribute(pcm_iter_kernel<KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    MMB_CUDA(cudaFuncSetAttribute(pcm_final_kernel<KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_set = true;
  }
  pcm_prep_kernel<<<P.nb, 128, 0, st>>>(S0, d, k, P.KP, P.DP, Yb[0], Sp[0], Sp[1], (P.nb + 7) & ~7);
  MMB_LAUNCH_CHECK("pcm_prep");
  // The iteration and final kernels are launched with programmatic stream serialisation: each
  // may begin (prologue only) while its predecessor is still running and synchronises with
  // griddepcontrol.wait before touching the predecessor's output.
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  for (int it = 0; it <= n_iter; ++it) {
    const int cur = it & 1;
    cfg.gridDim = dim3(P.nb);
    cfg.blockDim = dim3(kPcmThreads);
    cfg.dynamicSmemBytes = P.smem_iter;
    MMB_CUDA(cudaLaunchKernelEx(&cfg, pcm_iter_kernel<KMAX>, G, d, k, P.KP, P.DP, P.nb, (const double*)Yb[cur],
                                Yb[cur ^ 1], Qg, (const double*)Sp[cur], Sp[cur ^ 1], it == n_iter ? 2 : 1,
                                it == n_iter ? 1 : 0));
    count_launch("pcm_iter");
  }
  const int fin = (n_iter + 1) & 1;
  cfg.gridDim = dim3(1);
  cfg.blockDim = dim3(kPcmThreads);
  cfg.dynamicSmemBytes = P.smem_final;
  MMB_CUDA(cudaLaunchKernelEx(&cfg, pcm_final_kernel<KMAX>, d, k, P.KP, P.DP, P.nb, npc, transposed,
                              (const double*)Yb[fin], (const double*)Qg, (const double*)Sp[fin], pc));
  count_launch("pcm_final");
  return MMB_OK;
}

// S0 = X^T Omega for the N < d case (N tiny): thread per (column of X, column of Omega).
__global__ void start_block_xt_kernel(const float* __restrict__ X, int64_t N, int d,
                                      const double* __restrict__ Omega, int k, double* __restrict__ S0) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= d * k) return;
  const int c = idx % k, j = idx / k;
  double s = 0.0;
  for (int64_t n = 0; n < N; ++n) s = fma((double)X[n * d + j], Omega[n * k + c], s);
  S0[(size_t)j * k + c] = s;
}

}  // namespace mmb

using namespace mmb;

extern "C" size_t mmb_pc_workspace_bytes(int d, int k) { return pcm_plan(d, k).ws_bytes; }

extern "C" int mmb_pc_from_gram(const float* G, int d, const double* S0, int k, int npc,
                                int transposed, int n_iter, float* pc, void* ws, size_t ws_bytes,
                                mmb_stream_t stream) {
  MMB_REQUIRE(G && S0 && pc && ws, "null pointer");
  MMB_REQUIRE(d > 0 && d <= 512, "d must be in [1, 512]");
  MMB_REQUIRE(k > 0 && k <= kPcMaxK && npc > 0 && npc <= k, "need 0 < npc <= k <= 32");
  MMB_REQUIRE(ws_bytes >= mmb_pc_workspace_bytes(d, k), "workspace too small");
  MMB_REQUIRE(n_iter >= 0, "n_iter < 0");
  // The checks above keep every launch of the chain within its limits: d <= 512 and k <= 32 give
  // nb <= 64 CTAs (the partial sums read at most 64 slots), JS >= 5 j slices, and at most
  // 186,576 B of dynamic shared memory in pcm_iter_kernel and 162,008 B in pcm_final_kernel
  // (both under the 200 KiB pcm_run requests).
  return k <= 16 ? pcm_run<16>(G, d, S0, k, npc, transposed, n_iter, pc, (double*)ws, as_stream(stream))
                 : pcm_run<32>(G, d, S0, k, npc, transposed, n_iter, pc, (double*)ws, as_stream(stream));
}

extern "C" int mmb_start_block_xt(const float* X, int64_t N, int d, const double* Omega, int k,
                                  double* S0, mmb_stream_t stream) {
  MMB_REQUIRE(X && Omega && S0, "null pointer");
  MMB_REQUIRE(N > 0 && d > 0 && k > 0, "bad size");
  const int n = d * k;
  start_block_xt_kernel<<<(n + 127) / 128, 128, 0, as_stream(stream)>>>(X, N, d, Omega, k, S0);
  MMB_LAUNCH_CHECK("start_block_xt");
  return MMB_OK;
}
