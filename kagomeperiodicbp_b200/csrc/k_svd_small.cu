// Truncated SVD of a SMALL complex128 matrix entirely in one CTA's shared memory: one-sided (Hestenes)
// Jacobi on the rows of X = A (m <= n) or X = A^T (m > n), p = min(m, n) rows of length q = max(m, n),
// p*q*16 B <= ~220 KB.  This is the kernel behind every truncation at D = 2 and D = 3 (matrices up to
// 81 x 162) and behind the Rayleigh-Ritz stage of the subspace-iteration SVD that larger D uses
// (k_tsvd.cu) -- it replaces numpy.linalg.svd in mps.right_canonical (src/libs/bmpslib.py:733-772).
//
// One launch does the whole factorisation: load, sweeps until every pair's |<x_i,x_j>| / (|x_i||x_j|)
// is below tol (the convergence test stays on chip: no host round trip), rank sort, outputs.  A sweep is a
// round-robin tournament of pp-1 steps; in each step the pp/2 disjoint row pairs are rotated concurrently,
// one lane group (8/16/32 lanes, picked so that all pairs fit the 1024 threads) per pair: the group
// forms the 2x2 Gram matrix with shuffle reductions, builds the rotation in full double precision and
// applies it, writing the larger row first (de Rijk ordering, which also sorts the rows as a side effect).
//
// Outputs (same contract as the block-Jacobi kernel in k_svd.cu):
//   m <= n:  rows converge to s_i v_i^H ->  Vh_k = rows / s  (orthonormal to rounding),  US = A Vh_k^H
//   m >  n:  the rows carry an identity block behind them, [A^T | I], rotated along (Gram sums over the A^T part only):
//            rows converge to [s_i u_i^T | conj(v_i)^T]  ->  US_k = first part, Vh_k = conj(second part), both exact
// so US Vh is exactly the projection of A on the span found, whatever the rounding of the other factor.
#include "kbp_common.cuh"
#include "kbp_jacobi.cuh"
#include "kbp_ops.cuh"

#include <cooperative_groups.h>
#include <math.h>
#include <stdio.h>

namespace cg = cooperative_groups;

namespace kbp {

constexpr int SMALL_MAX_SWEEPS = 60;
constexpr size_t SMALL_SMEM_MAX = 225 * 1024;

struct SmallArgs {
  long long A, US, Vh;      // arena offsets; A is m x n with row stride lda
  int m, n, lda, keep;
  int nr_bulk, slot_lognorm, slot_trunc;
  int group;                // lanes per row pair
  const int* mask;          // per-chain predicate (kbp_ops.cuh: Arena::mask)
  int mask_want;
};

size_t svd_small_smem(int64_t m, int64_t n) {
  const int64_t p = m < n ? m : n, q = m <= n ? n : m + n;       // tall: rows of [A^T | I]
  return (size_t)(p * q) * sizeof(double2) + (size_t)p * (sizeof(double) + sizeof(int)) + 16 + (size_t)((p + 1) / 2) * sizeof(PairSums) + 64;
}

bool svd_small_fits(int64_t m, int64_t n) {
  const int64_t p = m < n ? m : n;
  return p <= 128 && svd_small_smem(m, n) <= SMALL_SMEM_MAX;
}

template <bool CACHED, int G>
__global__ void __launch_bounds__(CACHED ? 768 : 1024) svd_small_kernel(cplx* __restrict__ base, long long chain_stride, double* __restrict__ slots,
                                                                        int n_slots, SmallArgs g) {
  if (g.mask && g.mask[blockIdx.y] != g.mask_want) return;
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const int m = g.m, n = g.n;
  const bool mode_t = m > n;
  const int p = mode_t ? n : m, qx = mode_t ? m : n, q = mode_t ? m + n : n;   // q: row length incl. the identity block of a tall matrix
  cplx* X = reinterpret_cast<cplx*>(sm_raw);                                 // p x q
  double* s2 = reinterpret_cast<double*>(sm_raw + sizeof(cplx) * (size_t)p * q);   // p
  int* idx = reinterpret_cast<int*>(s2 + p);                                 // p
  PairSums* rec = reinterpret_cast<PairSums*>(sm_raw + ((sizeof(cplx) * (size_t)p * q + (size_t)p * 12 + 15) & ~(size_t)15));   // (p+1)/2 pair records
  __shared__ double red[34];

  cplx* cb = base + (long long)blockIdx.x * chain_stride;
  const cplx* A = cb + g.A;
  cplx* US = cb + g.US;
  cplx* Vh = cb + g.Vh;
  const int t = threadIdx.x, nt = blockDim.x, lane = t & 31, w = t >> 5, nw = nt >> 5;

  // ---- load (transposing when m > n) and ||A||_F^2
  double fro = 0.0;
  if (!mode_t) {
    for (int e = t; e < p * q; e += nt) {
      const int r = e / q, c = e - r * q;
      const cplx v = A[(long long)r * g.lda + c];
      X[e] = v;
      fro += cabs2(v);
    }
  } else {
    for (int e = t; e < m * n; e += nt) {           // coalesced read of A[r][c], scattered smem write
      const int r = e / n, c = e - r * n;
      const cplx v = A[(long long)r * g.lda + c];
      X[c * q + r] = v;
      fro += cabs2(v);
    }
    for (int e = t; e < n * n; e += nt) X[(e / n) * q + m + e % n] = cmake(e / n == e % n ? 1.0 : 0.0, 0.0);
  }
  const double fro2 = block_sum(fro, red);          // (contains the barrier that publishes X)
  const double floor2 = 1e-34 * fro2;

  // ---- Jacobi sweeps
  const int pp = (p + 1) & ~1, npairs = pp / 2;
  const int slot = t / G, gl = t - slot * G;
  // groups of one warp can take different branches (phantom row, dead rows): shuffles name their own group only
  const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
  const int cpl = (q + G - 1) / G;
  bool converged = p < 2;
#ifdef KBP_SMALL_DEBUG
  long long tstart = clock64();
#endif
  for (int sweep = 0; sweep < SMALL_MAX_SWEEPS && !converged; ++sweep) {
    bool big = false;
    PairWalk walk;
    walk.start(pp, slot);
    for (int step = 0; step < pp - 1; ++step) {
      int i, j;
      walk.get(step, i, j);
      if (slot < npairs && j < p) {
        cplx* xi = X + i * q;
        cplx* xj = X + j * q;
        if (CACHED) {
          switch (cpl) {
            case 1: jacobi_pair_cached<1, G>(xi, xj, q, qx, gl, gmask, floor2, big, rec + slot); break;
            case 2: jacobi_pair_cached<2, G>(xi, xj, q, qx, gl, gmask, floor2, big, rec + slot); break;
            case 3: jacobi_pair_cached<3, G>(xi, xj, q, qx, gl, gmask, floor2, big, rec + slot); break;
            case 4: jacobi_pair_cached<4, G>(xi, xj, q, qx, gl, gmask, floor2, big, rec + slot); break;
            case 5: jacobi_pair_cached<5, G>(xi, xj, q, qx, gl, gmask, floor2, big, rec + slot); break;
            default: jacobi_pair_cached<6, G>(xi, xj, q, qx, gl, gmask, floor2, big, rec + slot); break;
          }
        } else {
          double a = 0.0, b = 0.0, cr = 0.0, ci = 0.0;
          for (int c = gl; c < qx; c += G) {
            const cplx u = xi[c], v = xj[c];
            a = fma(u.x, u.x, fma(u.y, u.y, a));
            b = fma(v.x, v.x, fma(v.y, v.y, b));
            cr = fma(u.x, v.x, fma(u.y, v.y, cr));
            ci = fma(u.y, v.x, fma(-u.x, v.y, ci));
          }
          const double mine = group_reduce4<G>(a, b, cr, ci, gl, gmask);
          if (gl < 4) reinterpret_cast<double*>(rec + slot)[owner_pos(gl)] = mine;
          __syncwarp(gmask);
          const PairSums tot = rec[slot];
          Rotation R;
          if (make_rotation(tot.a, tot.b, tot.cr, tot.ci, floor2, big, R)) {
            for (int c = gl; c < q; c += G) {
              const cplx u = xi[c], v = xj[c];
              const double vr = R.er * v.x - R.ei * v.y, vi = R.er * v.y + R.ei * v.x;
              const cplx yi = make_double2(fma(R.cs, u.x, R.sn * vr), fma(R.cs, u.y, R.sn * vi));
              const cplx yj = make_double2(fma(R.cs, vr, -R.sn * u.x), fma(R.cs, vi, -R.sn * u.y));
              xi[c] = R.swap ? yj : yi;
              xj[c] = R.swap ? yi : yj;
            }
          }
        }
      }
      walk.next();
      __syncthreads();
    }
    // One-sided Jacobi converges quadratically at the end: once every pair of a sweep started with cos^2 <= tol, the next
    // sweep would find nothing to do -- skip it.  (`big`: some pair of this sweep was above that.)
    converged = !__syncthreads_or(big ? 1 : 0);
#ifdef KBP_SMALL_DEBUG
    if (t == 0) printf("[small %dx%d] sweep %d converged %d  cycles %lld\n", p, q, sweep, (int)converged, clock64() - tstart);
#endif
  }

  // ---- singular values = row norms, rank sort (descending, stable)
  for (int i = w; i < p; i += nw) {
    double acc = 0.0;
    const cplx* row = X + i * q;
    for (int c = lane; c < qx; c += 32) acc += cabs2(row[c]);
    acc = warp_sum(acc);
    if (lane == 0) s2[i] = (acc == acc && acc < 1e300) ? acc : 0.0;
  }
  for (int k = t; k < p; k += nt) idx[k] = k;       // identity first: non-finite input can never index out of bounds
  __syncthreads();
  double disc_part = 0.0;
  for (int i = t; i < p; i += nt) {
    const double si = s2[i];
    int rank = 0;
    for (int j = 0; j < p; ++j) {
      const double sj = s2[j];
      rank += (sj > si) || (sj == si && j < i);
    }
    if (rank >= g.keep) disc_part += si;        // summed directly: total - kept would cancel
    idx[rank] = i;
  }
  const double disc = block_sum(disc_part, red);
  const double frob = sqrt(fro2);
  const double scale = (g.nr_bulk && frob > 0.0) ? 1.0 / frob : 1.0;
  const int keep = g.keep;
  if (!mode_t) {
    // Vh_k = rows / s ;  US = A Vh_k^H  (A re-read from global memory: X was overwritten)
    for (int e = t; e < keep * n; e += nt) {
      const int k = e / n, c = e - k * n;
      const double sk2 = s2[idx[k]];
      Vh[e] = sk2 > floor2 ? cscale(X[idx[k] * q + c], rsqrt(sk2)) : cmake(0.0, 0.0);
    }
    for (int e = w; g.US >= 0 && e < m * keep; e += nw) {
      const int r = e / keep, k = e - r * keep;
      const double sk2 = s2[idx[k]];
      const cplx* xr = X + idx[k] * q;
      const cplx* ar = A + (long long)r * g.lda;
      cplx acc = cmake(0.0, 0.0);
      for (int c = lane; c < n; c += 32) acc = cadd(acc, cmulc(ar[c], xr[c]));
      acc = warp_sum(acc);
      if (lane == 0) US[e] = sk2 > floor2 ? cscale(acc, rsqrt(sk2) * scale) : cmake(0.0, 0.0);
    }
  } else {
    // US_k = data part of the rows ;  Vh_k = conj of the accumulated-rotation part (orthonormal to rounding)
    for (int e = t; g.US >= 0 && e < m * keep; e += nt) {
      const int r = e / keep, k = e - r * keep;
      US[e] = cscale(X[idx[k] * q + r], scale);
    }
    for (int e = t; e < keep * n; e += nt) {
      const int k = e / n, c = e - k * n;
      Vh[e] = s2[idx[k]] > floor2 ? cconj(X[idx[k] * q + m + c]) : cmake(0.0, 0.0);
    }
  }
  if (t == 0) {
    double* sl = slots + (long long)blockIdx.x * n_slots;
    if (g.nr_bulk && g.slot_lognorm >= 0 && frob > 0.0) sl[g.slot_lognorm] += log(frob);
    if (g.slot_trunc >= 0 && fro2 > 0.0) sl[g.slot_trunc] += sqrt(disc / fro2);
    if (!converged) sl[n_slots - 1] += 1.0;        // engine-reserved status slot: Jacobi did not converge
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// The same factorisation on a thread-block CLUSTER: the one-CTA kernel above is bound by the FP64 rate of a single SM
// (all pp/2 pair rotations of a step run there).  Here C CTAs (C SMs) share one matrix by COLUMNS: CTA r keeps columns
// [r ql, (r+1) ql) of every row in its shared memory.  A step is
//   partial Gram sums of each pair over the local columns -> pushed into every CTA's shared memory (DSMEM stores)
//   -> one cluster barrier -> every CTA adds the C partials in rank order (bitwise identical totals, so all CTAs take
//   the same decisions and build the same rotation) -> rotates its own columns.
// Per-SM arithmetic drops ~C-fold for the sums and the updates; the rotation itself (three special-function chains) is
// recomputed everywhere.  The price is one cluster barrier (~400 cycles) + 32 B x pairs x C of DSMEM traffic per step.
constexpr int CL_C = 4;     // CTAs per cluster
constexpr int CL_G = 8;     // lanes per row pair
constexpr int CL_MIN_P = 48; // smallest p that takes the cluster kernel

// The per-step exchange does not use the cluster barrier (its release fence costs ~900 cycles per step here): partial sums
// travel as asynchronous DSMEM stores that complete a transaction count on the RECEIVER's mbarrier (st.async ...
// mbarrier::complete_tx::bytes; SASS: STAS + SYNCS), and each CTA waits on its own mbarrier only.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t map_to_rank(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_async_2f64(uint32_t remote_addr, double x, double y, uint32_t remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];"
               :: "r"(remote_addr), "d"(x), "d"(y), "r"(remote_bar) : "memory");
}
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (int spins = 0; !done && spins < (1 << 20); ++spins)
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  return done != 0;
}

template <int CPL, int G>
__global__ void __launch_bounds__(1024) svd_cluster_kernel(cplx* __restrict__ base, long long chain_stride, double* __restrict__ slots,
                                                           int n_slots, SmallArgs g) {
  if (g.mask && g.mask[blockIdx.y] != g.mask_want) return;
  constexpr int C = CL_C;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const int m = g.m, n = g.n;
  const bool mode_t = m > n;
  const int p = mode_t ? n : m, qx = mode_t ? m : n, q = mode_t ? m + n : n;
  const int ql = (q + C - 1) / C, c0 = rank * ql;                       // this CTA's column slice [c0, c0 + qn)
  const int ld = ql | 1;                                                // odd row stride: rows start in different banks
  const int qn = max(0, min(ql, q - c0)), qxn = max(0, min(qn, qx - c0));     // qxn: local columns that are data (enter the Gram sums)
  const int pp = (p + 1) & ~1, npairs = pp / 2;
  cplx* X = reinterpret_cast<cplx*>(sm_raw);                                    // p x ld
  PairSums* part = reinterpret_cast<PairSums*>(sm_raw + sizeof(cplx) * (size_t)p * ld);   // [2][C][npairs]
  PairSums* rec = part + 2 * C * npairs;                                        // [npairs] this CTA's own sums of the current step
  double* s2p = reinterpret_cast<double*>(rec + npairs);                        // [C][p]
  double* s2 = s2p + C * p;                                                     // p
  int* idx = reinterpret_cast<int*>(s2 + p);                                    // p
  __shared__ double red[34];
  __shared__ __align__(8) unsigned long long bar[2];                            // one mbarrier per exchange buffer

  cplx* cb = base + (long long)blockIdx.y * chain_stride;
  const cplx* A = cb + g.A;
  cplx* US = cb + g.US;
  cplx* Vh = cb + g.Vh;
  const int t = threadIdx.x, nt = blockDim.x, lane = t & 31, w = t >> 5, nw = nt >> 5;

  // ---- load this CTA's columns; ||A||_F^2 over the whole matrix in every CTA (same order -> same value everywhere)
  if (!mode_t) {
    for (int e = t; e < p * qn; e += nt) {
      const int r = e / qn, cl = e - r * qn;
      X[r * ld + cl] = A[(long long)r * g.lda + c0 + cl];
    }
  } else {
    for (int e = t; e < p * qn; e += nt) {
      const int cl = e / p, r = e - cl * p, c = c0 + cl;                    // row r of X = column r of A, then row r of I
      X[r * ld + cl] = c < m ? A[(long long)c * g.lda + r] : cmake(c - m == r ? 1.0 : 0.0, 0.0);
    }
  }
  double fro = 0.0;
  for (int e = t; e < m * n; e += nt) fro += cabs2(A[(long long)(e / n) * g.lda + e % n]);
  const double fro2 = block_sum(fro, red);
  const double floor2 = 1e-34 * fro2;

  const int slot = t / G, gl = t - slot * G;
  const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
  // where lane gl < C delivers this CTA's partial sums: CTA gl's copy of part[.][rank][slot], completing CTA gl's mbarrier
  const uint32_t remote_part = map_to_rank(smem_u32(part + rank * npairs + (slot < npairs ? slot : 0)), gl < C ? gl : 0);
  const uint32_t remote_bar = map_to_rank(smem_u32(&bar[0]), gl < C ? gl : 0);
  const uint32_t bar0 = smem_u32(&bar[0]);
  const uint32_t step_bytes = (uint32_t)(C * (p / 2) * sizeof(PairSums));   // p/2 real pairs per step, from each of the C CTAs
  if (t == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar0));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar0 + 8));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  bool converged = p < 2, lost = false;
  int tick = 0;
  uint32_t parity = 0;                              // bit k: phase parity of bar[k]
#ifdef KBP_SMALL_DEBUG
  long long tstart = clock64();
  long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif
  cluster.sync();                                   // every CTA of the cluster is resident before the first remote store
  for (int sweep = 0; sweep < SMALL_MAX_SWEEPS && !converged && !lost; ++sweep) {
    bool big = false;
    PairWalk walk;
    walk.start(pp, slot);
    for (int step = 0; step < pp - 1; ++step) {
#ifdef KBP_SMALL_DEBUG
      const long long k0 = clock64();
#endif
      if (t == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar0 + 8 * tick), "r"(step_bytes) : "memory");
      int i, j;
      walk.get(step, i, j);
      const bool act = slot < npairs && j < p;
#ifdef KBP_SMALL_DEBUG
      const long long q0 = clock64();
      long long q1 = q0, q2 = q0;
#endif
      cplx u[CPL], v[CPL];
      cplx* xi = X + i * ld;
      cplx* xj = X + j * ld;
      if (act) {
        double a = 0.0, b = 0.0, cr = 0.0, ci = 0.0;
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          const int cl = gl + k * G;
          u[k] = cl < qn ? xi[cl] : cmake(0.0, 0.0);
          v[k] = cl < qn ? xj[cl] : cmake(0.0, 0.0);
          if (cl < qxn) {
            a = fma(u[k].x, u[k].x, fma(u[k].y, u[k].y, a));
            b = fma(v[k].x, v[k].x, fma(v[k].y, v[k].y, b));
            cr = fma(u[k].x, v[k].x, fma(u[k].y, v[k].y, cr));
            ci = fma(u[k].y, v[k].x, fma(-u[k].x, v[k].y, ci));
          }
        }
#ifdef KBP_SMALL_DEBUG
        q1 = clock64() + (long long)(a * 0.0);
#endif
        const double mine = group_reduce4<G>(a, b, cr, ci, gl, gmask);
#ifdef KBP_SMALL_DEBUG
        q2 = clock64() + (long long)(mine * 0.0);
#endif
        if (gl < 4) reinterpret_cast<double*>(rec + slot)[owner_pos(gl)] = mine;
        __syncwarp(gmask);
        if (gl < C) {
          const PairSums ps = rec[slot];
          const uint32_t dst = remote_part + (uint32_t)(tick * C * npairs * sizeof(PairSums));
          st_async_2f64(dst, ps.a, ps.b, remote_bar + 8 * tick);
          st_async_2f64(dst + 16, ps.cr, ps.ci, remote_bar + 8 * tick);
        }
      }
#ifdef KBP_SMALL_DEBUG
      const long long k1 = clock64();
#endif
      if (!mbar_wait(bar0 + 8 * tick, (parity >> tick) & 1u)) lost = true;      // (never in a healthy run: bounded spin instead of a hang)
      parity ^= 1u << tick;
#ifdef KBP_SMALL_DEBUG
      const long long k2 = clock64();
#endif
      if (act) {
        const PairSums* ps = part + tick * C * npairs + slot;
        double a = 0.0, b = 0.0, cr = 0.0, ci = 0.0;
#pragma unroll
        for (int r = 0; r < C; ++r) { a += ps[r * npairs].a; b += ps[r * npairs].b; cr += ps[r * npairs].cr; ci += ps[r * npairs].ci; }
        Rotation R;
        if (make_rotation(a, b, cr, ci, floor2, big, R)) {
#pragma unroll
          for (int k = 0; k < CPL; ++k) {
            const int cl = gl + k * G;
            if (cl < qn) {
              const double vr = R.er * v[k].x - R.ei * v[k].y, vi = R.er * v[k].y + R.ei * v[k].x;
              const cplx yi = make_double2(fma(R.cs, u[k].x, R.sn * vr), fma(R.cs, u[k].y, R.sn * vi));
              const cplx yj = make_double2(fma(R.cs, vr, -R.sn * u[k].x), fma(R.cs, vi, -R.sn * u[k].y));
              xi[cl] = R.swap ? yj : yi;
              xj[cl] = R.swap ? yi : yj;
            }
          }
        }
      }
      tick ^= 1;
      walk.next();
#ifdef KBP_SMALL_DEBUG
      const long long k3 = clock64();
#endif
      __syncthreads();
#ifdef KBP_SMALL_DEBUG
      const long long k4 = clock64();
      ph[0] += k1 - k0; ph[1] += k2 - k1; ph[2] += k3 - k2; ph[3] += k4 - k3;
      ph[4] += q0 - k0; ph[5] += q1 - q0; ph[6] += q2 - q1; ph[7] += k1 - q2;
#endif
    }
    converged = !__syncthreads_or(big ? 1 : 0);     // identical in every CTA: same totals, same decisions
    lost = __syncthreads_or(lost ? 1 : 0) != 0;
#ifdef KBP_SMALL_DEBUG
    if (t == 0 && rank == 0) printf("[cluster %dx%d C %d G %d] sweep %d converged %d  cycles %lld  phases: dots %lld barrier %lld rotate %lld sync %lld | expect+walk %lld load+fma %lld shuffles %lld send %lld\n", p, q, C, G, sweep, (int)converged, clock64() - tstart, ph[0], ph[1], ph[2], ph[3], ph[4], ph[5], ph[6], ph[7]);
#endif
  }

  // ---- singular values: partial row norms -> every CTA, summed in rank order
  for (int i = w; i < p; i += nw) {
    double acc = 0.0;
    const cplx* row = X + i * ld;
    for (int cl = lane; cl < qxn; cl += 32) acc += cabs2(row[cl]);
    acc = warp_sum(acc);
    if (lane < C) *cluster.map_shared_rank(s2p + rank * p + i, lane) = acc;
  }
  cluster.sync();
  for (int i = t; i < p; i += nt) {
    double acc = 0.0;
    for (int r = 0; r < C; ++r) acc += s2p[r * p + i];
    s2[i] = (acc == acc && acc < 1e300) ? acc : 0.0;
    idx[i] = i;
  }
  __syncthreads();
  double disc_part = 0.0;
  for (int i = t; i < p; i += nt) {
    const double si = s2[i];
    int rk = 0;
    for (int j = 0; j < p; ++j) {
      const double sj = s2[j];
      rk += (sj > si) || (sj == si && j < i);
    }
    if (rk >= g.keep) disc_part += si;
    idx[rk] = i;
  }
  const double disc = block_sum(disc_part, red);
  const double frob = sqrt(fro2);
  const double scale = (g.nr_bulk && frob > 0.0) ? 1.0 / frob : 1.0;
  const int keep = g.keep;
  if (!mode_t) {
    for (int e = t; e < keep * qn; e += nt) {
      const int k = e / qn, cl = e - k * qn;
      const double sk2 = s2[idx[k]];
      Vh[(long long)k * n + c0 + cl] = sk2 > floor2 ? cscale(X[idx[k] * ld + cl], rsqrt(sk2)) : cmake(0.0, 0.0);
    }
    if (g.US >= 0) {
      // US = A Vh_k^H needs whole rows of Vh: publish them, then CTA r takes the rows r, r + C, ... of US
      __threadfence();
      cluster.sync();
      for (int e = w; e < m * keep; e += nw) {
        const int r = e / keep, k = e - r * keep;
        if (r % C != rank) continue;
        const cplx* ar = A + (long long)r * g.lda;
        const cplx* vr = Vh + (long long)k * n;
        cplx acc = cmake(0.0, 0.0);
        for (int c = lane; c < n; c += 32) acc = cadd(acc, cmulc(ar[c], __ldcg(vr + c)));
        acc = warp_sum(acc);
        if (lane == 0) US[e] = cscale(acc, scale);
      }
    }
  } else {
    for (int e = t; e < keep * qn; e += nt) {
      const int k = e / qn, cl = e - k * qn, c = c0 + cl;
      const cplx x = X[idx[k] * ld + cl];
      if (c < m) { if (g.US >= 0) US[(long long)c * keep + k] = cscale(x, scale); }
      else Vh[(long long)k * n + (c - m)] = s2[idx[k]] > floor2 ? cconj(x) : cmake(0.0, 0.0);
    }
  }
  if (t == 0 && rank == 0) {
    double* sl = slots + (long long)blockIdx.y * n_slots;
    if (g.nr_bulk && g.slot_lognorm >= 0 && frob > 0.0) sl[g.slot_lognorm] += log(frob);
    if (g.slot_trunc >= 0 && fro2 > 0.0) sl[g.slot_trunc] += sqrt(disc / fro2);
    if (!converged || lost) sl[n_slots - 1] += 1.0;
  }
}

template <int CPL, int G>
static cudaError_t launch_cluster(const Arena& a, const SmallArgs& g, int C, int threads, size_t smem) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)C, (unsigned)a.nb);
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = a.stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)C;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, svd_cluster_kernel<CPL, G>, a.base, (long long)a.chain_stride, a.slots, a.n_slots, g);
}

void svd_small(const Arena& a, int64_t A, int64_t lda, int64_t US, int64_t Vh, int64_t m, int64_t n, int64_t keep, int nr_bulk,
               int slot_lognorm, int slot_trunc) {
  SmallArgs g;
  g.mask = a.mask; g.mask_want = a.mask_want;
  g.A = A; g.US = US; g.Vh = Vh; g.m = (int)m; g.n = (int)n; g.lda = (int)lda; g.keep = (int)keep;
  g.nr_bulk = nr_bulk; g.slot_lognorm = slot_lognorm; g.slot_trunc = slot_trunc;
  const int p = (int)(m < n ? m : n), pp = (p + 1) & ~1, npairs = pp / 2 > 0 ? pp / 2 : 1;
  const int q = (int)(m <= n ? n : m + n);
  if (p >= CL_MIN_P) {                              // cluster version for the larger matrices
    // (4 and 2 lanes per pair were measured slower: the per-lane FP64 work grows faster than the shuffles shrink)
    const int C = CL_C, ql = (q + C - 1) / C, Gc = CL_G;
    const int cpl = (ql + Gc - 1) / Gc;
    if (cpl <= 6 && npairs * Gc <= 1024) {
      g.group = Gc;
      int threads = (npairs * Gc + 31) / 32 * 32;
      if (threads < 64) threads = 64;
      const size_t smem = sizeof(double2) * (size_t)p * (ql | 1) + sizeof(PairSums) * (2 * (size_t)C + 1) * npairs +
                          sizeof(double) * ((size_t)C * p + p) + sizeof(int) * (size_t)p + 64;
      cudaError_t e = cudaErrorInvalidValue;
#define KBP_CL(CP, GG) if (cpl == CP && Gc == GG) e = launch_cluster<CP, GG>(a, g, C, threads, smem)
      KBP_CL(1, 8); KBP_CL(2, 8); KBP_CL(3, 8); KBP_CL(4, 8); KBP_CL(5, 8); KBP_CL(6, 8);
#undef KBP_CL
      if (e == cudaSuccess) { ++*a.launches; return; }
      cudaGetLastError();                           // cluster launch refused: use the one-CTA kernel
    }
  }
  int G = 32;
  while (G > 8 && npairs * G > 1024) G >>= 1;
  g.group = G;
  int threads = npairs * G;
  threads = (threads + 31) / 32 * 32;
  if (threads < 256) threads = 256;
  if (threads > 1024) threads = 1024;
  const bool cached = threads <= 768 && (q + G - 1) / G <= 6;
  const size_t smem = svd_small_smem(m, n);
#define KBP_SMALL_LAUNCH(CA, GG) svd_small_kernel<CA, GG><<<a.nb, threads, smem, a.stream>>>(a.base, a.chain_stride, a.slots, a.n_slots, g)
  if (G == 32) { if (cached) KBP_SMALL_LAUNCH(true, 32); else KBP_SMALL_LAUNCH(false, 32); }
  else if (G == 16) { if (cached) KBP_SMALL_LAUNCH(true, 16); else KBP_SMALL_LAUNCH(false, 16); }
  else { if (cached) KBP_SMALL_LAUNCH(true, 8); else KBP_SMALL_LAUNCH(false, 8); }
#undef KBP_SMALL_LAUNCH
  ++*a.launches;
}

void init_svd_small_attributes() {
  cudaFuncSetAttribute(svd_small_kernel<false, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_small_kernel<true, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_small_kernel<false, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_small_kernel<true, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_small_kernel<false, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_small_kernel<true, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_cluster_kernel<1, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_cluster_kernel<2, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_cluster_kernel<3, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_cluster_kernel<4, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_cluster_kernel<5, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
  cudaFuncSetAttribute(svd_cluster_kernel<6, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMALL_SMEM_MAX);
}

}  // namespace kbp
