// Batched truncated SVD of complex128 matrices by block one-sided Jacobi (Hestenes) -- the kernel
// that replaces the reference's numpy.linalg.svd inside right_canonical (src/libs/bmpslib.py:733-772),
// where >= 60 % of its wall time goes.
//
// Work matrix Z (p_pad x LD, row-major), rows = the vectors being orthogonalised:
//     Z = [ X | J ],   X = A^T (m >= n, "mode T")  or  X = A (m < n, "mode N"),   J = I  (accumulates the rotations)
// so p = min(m, n) vectors of length q = max(m, n).  Rows are grouped in blocks of 16; one sweep visits
// all block pairs in a round-robin tournament (nblk-1 rounds of nblk/2 independent pairs, one CTA per
// pair and chain, one launch per round).  Per pair:
//   1. Gram  G = P P^H  (32 x 32) over the X columns                 -- DMMA (FP64 tensor pipe)
//   2. Hermitian Jacobi eigensolve  G = W L W^H  in shared memory, eigenvalues sorted descending
//   3. rotate the 32 rows:  P <- W^H P  over all LD columns (X and J)  -- DMMA
// A pair whose largest |G_ij| / sqrt(G_ii G_jj) is below tol is left alone; a sweep in which every
// pair was left alone ends the iteration (one pinned-memory flag read per sweep).  After convergence
// the rows of X are mutually orthogonal:  A = J^H diag(s) Yhat  (mode N)  or  A = Yhat^T diag(s) conj(J)
// (mode T), with s_i the row norms; the extraction kernel sorts s, keeps the largest `keep`, and
// writes U_k diag(s_k) and V_k^H -- in mode T without ever dividing by a singular value.
#include "kbp_common.cuh"
#include "kbp_ops.cuh"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>

namespace kbp {

constexpr int JB = 16;        // rows per block
constexpr int PR = 2 * JB;    // rows per pair
constexpr int KC = 32;        // columns staged per Gram step
constexpr int LDP = KC + 4;   // shared row stride (doubles): 36 mod 16 == 4 -> conflict-free fragments
constexpr size_t SVD_ROUND_SMEM = 3 * sizeof(double2) * PR * (PR + 1) + 2 * sizeof(double) * PR * LDP;
constexpr double SVD_TOL = 1e-14;
constexpr int SVD_MAX_SWEEPS = 40;
constexpr int SVD_INNER_LO = 2;          // inner Jacobi sweeps of a block pair during the first 24 outer sweeps (15 after)

static inline int64_t round_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

struct SvdGeom {
  int mode_t;           // 1: X = A^T, 0: X = A
  int m, n, p, q;
  int p_pad, q_pad, ld;
  int nblk;
};

static SvdGeom svd_geom(int64_t m, int64_t n) {
  SvdGeom g;
  g.m = (int)m; g.n = (int)n;
  g.mode_t = m >= n;
  g.p = (int)(m >= n ? n : m);
  g.q = (int)(m >= n ? m : n);
  g.p_pad = (int)round_up(g.p, PR);
  g.q_pad = (int)round_up(g.q, 8);
  g.ld = g.q_pad + g.p_pad;
  g.nblk = g.p_pad / JB;
  return g;
}

int64_t tsvd_work_elems(int64_t m, int64_t n);
int tsvd_block(int64_t m, int64_t n, int64_t keep);
bool svd_small_fits(int64_t m, int64_t n);
void svd_small(const Arena& a, int64_t A, int64_t lda, int64_t US, int64_t Vh, int64_t m, int64_t n, int64_t keep, int nr_bulk,
               int slot_lognorm, int slot_trunc);
int svd_truncate_subspace(const Arena& a, int64_t A, int64_t US, int64_t Vh, int64_t work, int64_t m, int64_t n, int64_t keep,
                          int nr_bulk, int slot_lognorm, int slot_trunc, int b);
void phase_fix(const Arena& a, int64_t Vh, int64_t US, int64_t m, int64_t n, int64_t keep, int us_too);


int64_t svd_work_elems(int64_t m, int64_t n) {
  SvdGeom g = svd_geom(m, n);
  const int64_t jac = (int64_t)g.p_pad * g.ld, sub = tsvd_work_elems(m, n);
  return jac > sub ? jac : sub;
}

// ------------------------------------------------------------------------------------------------
__global__ void svd_init_kernel(cplx* __restrict__ base, long long chain_stride, long long A_, long long Z_, SvdGeom g,
                                const int* __restrict__ mask, int mask_want) {
  if (mask && mask[blockIdx.y] != mask_want) return;
  cplx* cb = base + (long long)blockIdx.y * chain_stride;
  const cplx* A = cb + A_;
  cplx* Z = cb + Z_;
  const long long total = (long long)g.p_pad * g.ld;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    int i = (int)(e / g.ld), c = (int)(e % g.ld);
    cplx v = cmake(0.0, 0.0);
    if (c < g.q_pad) {
      if (i < g.p && c < g.q) v = g.mode_t ? A[(long long)c * g.n + i] : A[(long long)i * g.n + c];
    } else if (c - g.q_pad == i) {
      v = cmake(1.0, 0.0);
    }
    Z[e] = v;
  }
}

// round-robin tournament: players 0..n-1 (n even), round r in [0, n-1), table t in [0, n/2)
__device__ __forceinline__ void rr_pair(int n, int r, int t, int& a, int& b) {
  const int m = n - 1;
  if (t == 0) { a = m; b = r; }
  else { a = (r + t) % m; b = (r - t + m) % m; }
  if (a > b) { int x = a; a = b; b = x; }
}

// Hermitian 2x2 Jacobi rotation for the pair (a, b): R = [[c, s], [-s e, c e]], e = exp(-i arg g_ab).
// The dependent FP64 chain is the cost of a Jacobi step, so it is kept to two rsqrt: 1/|g_ab| (needed to
// double precision: |e| must be 1) and 1/sqrt(1+t^2) (c^2+s^2 must be 1); tan(theta) itself only steers
// the rotation and is evaluated in single precision -- the pair's off-diagonal drops by ~1e-7 per visit
// instead of to zero, which the cyclic iteration absorbs.  Returns false (identity) for dead / tiny pairs.
__device__ __forceinline__ bool jacobi_rot(double gaa, double gbb, cplx gab, double floor2, double& c, double& s, cplx& e) {
  c = 1.0; s = 0.0; e = cmake(1.0, 0.0);
  const double r2 = cabs2(gab);
  if (!(gaa > floor2 && gbb > floor2) || !(r2 > 1e-34 * gaa * gbb)) return false;
  const double inv_ab = rsqrt(r2);
  const double ab2 = 2.0 * r2 * inv_ab, delta = gbb - gaa;
  // tan(theta) = 2|g_ab| sgn(delta) / (|delta| + sqrt(delta^2 + 4|g_ab|^2)), operands brought into float range by
  // a common power of two (live pairs have |g_ab|/|delta| >= 1e-34, so nothing underflows)
  const int ex = ilogb(fmax(fabs(delta), ab2));
  const float df = (float)scalbn(delta, -ex), af = (float)scalbn(ab2, -ex);
  float tf = af / (fabsf(df) + sqrtf(fmaf(df, df, af * af)));
  tf = copysignf(tf, df);
  const double tt = (double)tf;
  c = rsqrt(fma(tt, tt, 1.0));
  s = tt * c;
  e = cmake(gab.x * inv_ab, -gab.y * inv_ab);
  return true;
}

__device__ __forceinline__ unsigned long long dbl_bits_nonneg(double x) { return (unsigned long long)__double_as_longlong(x); }

__global__ void __launch_bounds__(256) svd_round_kernel(cplx* __restrict__ base, long long chain_stride, long long Z_, SvdGeom g,
                                                        int round, double tol, const double* __restrict__ off_prev,
                                                        double* __restrict__ off_cur, const double* __restrict__ fro2, int inner_lo,
                                                        const SvdCtl* __restrict__ ctl) {
  // shared: staged operand planes (phase 1) reused as W^H planes (phase 3); G and W for the eigensolve
  extern __shared__ __align__(16) unsigned char svd_smem[];
  cplx (*Gs)[PR + 1] = reinterpret_cast<cplx (*)[PR + 1]>(svd_smem);
  cplx (*Ws)[PR + 1] = reinterpret_cast<cplx (*)[PR + 1]>(svd_smem + sizeof(cplx) * PR * (PR + 1));
  cplx (*G2)[PR + 1] = reinterpret_cast<cplx (*)[PR + 1]>(svd_smem + 2 * sizeof(cplx) * PR * (PR + 1));
  double (*Ps_re)[LDP] = reinterpret_cast<double (*)[LDP]>(svd_smem + 3 * sizeof(cplx) * PR * (PR + 1));
  double (*Ps_im)[LDP] = reinterpret_cast<double (*)[LDP]>(svd_smem + 3 * sizeof(cplx) * PR * (PR + 1) + sizeof(double) * PR * LDP);
  __shared__ double sh_red[34];
  __shared__ int perm[PR];

  const int chain = blockIdx.y;
  if (off_prev[chain] < tol) return;            // this chain converged in the previous sweep (or takes no part)
  const int inner_max = ctl->sweeps < 24 ? inner_lo : 15;
  // rows whose norm is below 1e-17 ||A||_F are rounding residue of exactly dependent rows: treated as zero
  const double floor2 = 1e-34 * fro2[chain];
  cplx* Z = base + (long long)chain * chain_stride + Z_;
  int bi, bj;
  rr_pair(g.nblk, round, blockIdx.x, bi, bj);
  const int t = threadIdx.x, lane = t & 31, w = t >> 5, gq = lane >> 2, q = lane & 3;
  const int ld = g.ld;
  auto grow = [&](int k) -> long long { return (long long)(k < JB ? bi * JB + k : bj * JB + (k - JB)) * ld; };

  // ---------------- phase 1: G = P P^H over the X columns (DMMA) ----------------
  const int mt = w & 1, ntile = w >> 1;          // warp's 16x8 tile of the 32x32 Gram matrix
  double gr[4] = {0, 0, 0, 0}, gi[4] = {0, 0, 0, 0};
  cplx stage[4];
  const int sc = t & 31, sr = t >> 5;            // staging: column sc, rows sr + 8*r
  auto fetch = [&](int c0) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int c = c0 + sc;
      stage[r] = c < g.q_pad ? Z[grow(sr + 8 * r) + c] : cmake(0.0, 0.0);
    }
  };
  fetch(0);
  for (int c0 = 0; c0 < g.q_pad; c0 += KC) {
#pragma unroll
    for (int r = 0; r < 4; ++r) { Ps_re[sr + 8 * r][sc] = stage[r].x; Ps_im[sr + 8 * r][sc] = stage[r].y; }
    __syncthreads();
    if (c0 + KC < g.q_pad) fetch(c0 + KC);
#pragma unroll
    for (int ks = 0; ks < KC / 8; ++ks) {
      double ar[4], ai[4], an[4], br[2], bim[2];
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int rr = mt * 16 + gq + 8 * (v & 1), kk = ks * 8 + q + 4 * (v >> 1);
        ar[v] = Ps_re[rr][kk]; ai[v] = Ps_im[rr][kk]; an[v] = -ar[v];
      }
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        const int rr = ntile * 8 + gq, kk = ks * 8 + q + 4 * v;
        br[v] = Ps_re[rr][kk]; bim[v] = Ps_im[rr][kk];
      }
      // (ar + i ai)(br - i bi): re = ar br + ai bi, im = ai br - ar bi
      dmma16x8x8(gr, ar, br);
      dmma16x8x8(gr, ai, bim);
      dmma16x8x8(gi, ai, br);
      dmma16x8x8(gi, an, bim);
    }
    __syncthreads();
  }
#pragma unroll
  for (int v = 0; v < 4; ++v) Gs[mt * 16 + gq + 8 * (v >> 1)][ntile * 8 + 2 * q + (v & 1)] = cmake(gr[v], gi[v]);
  __syncthreads();

  // ---------------- convergence measure of this pair ----------------
  double off = 0.0;
  for (int e = t; e < PR * PR; e += 256) {
    const int i = e / PR, j = e % PR;
    if (i < j) {
      const double gi_ = Gs[i][i].x, gj_ = Gs[j][j].x;
      if (gi_ > floor2 && gj_ > floor2) off = fmax(off, sqrt(cabs2(Gs[i][j]) / (gi_ * gj_)));
    }
  }
  off = warp_max(off);
  if (lane == 0) sh_red[w] = off;
  __syncthreads();
  if (t < 32) {
    double x = t < 8 ? sh_red[t] : 0.0;
    x = warp_max(x);
    if (t == 0) sh_red[33] = x;
  }
  __syncthreads();
  off = sh_red[33];
  if (t == 0) atomicMax(reinterpret_cast<unsigned long long*>(off_cur + chain), dbl_bits_nonneg(off));
  if (off < tol) return;

  // ---------------- phase 2: Hermitian Jacobi eigensolve of G (shared memory) ----------------
  // Parallel-ordered cyclic Jacobi: 31 steps of 16 disjoint rotations per sweep.  Thread (pr, qc) owns the
  // 2x2 block rows{a_pr,b_pr} x cols{a_qc,b_qc}: it recomputes the two rotations it needs from the old G,
  // applies R_pr^H . block . R_qc from buffer `cur` into buffer `cur^1`, and rotates its 2x2 block of W in
  // place -- ONE barrier per step.  The solve stops once the largest |g_ab|/sqrt(g_aa g_bb) seen in a sweep is
  // below max(2e-15, 1e-3 off^2): the residual it leaves is what the next outer sweep starts from, and
  // the outer iteration converges quadratically, so early outer sweeps need no 1e-15 inner solve.
  for (int e = t; e < PR * PR; e += 256) Ws[e / PR][e % PR] = (e / PR == e % PR) ? cmake(1.0, 0.0) : cmake(0.0, 0.0);
  const double inner_tol = fmax(2e-15, 1e-3 * off * off);
  int cur = 0;
  const int pr = t >> 4, qc = t & 15;
  __syncthreads();
  for (int isweep = 0; isweep < inner_max; ++isweep) {
    double my_off2 = 0.0;
    for (int step = 0; step < PR - 1; ++step) {
      cplx (*Go)[PR + 1] = cur ? G2 : Gs;
      cplx (*Gn)[PR + 1] = cur ? Gs : G2;
      int ap, bp, aq, bq;
      rr_pair(PR, step, pr, ap, bp);
      rr_pair(PR, step, qc, aq, bq);
      double cp, sp, cq, sq;
      cplx ep, eq;
      jacobi_rot(Go[ap][ap].x, Go[bp][bp].x, Go[ap][bp], floor2, cp, sp, ep);
      {
        const double gaa = Go[aq][aq].x, gbb = Go[bq][bq].x;
        const cplx gab = Go[aq][bq];
        if (jacobi_rot(gaa, gbb, gab, floor2, cq, sq, eq) && pr == qc) my_off2 = fmax(my_off2, cabs2(gab) / (gaa * gbb));
      }
      // column rotation R_q = [[c, s], [-s e, c e]] on columns (aq, bq), then row rotation R_p^H on rows (ap, bp)
      const cplx x00 = Go[ap][aq], x01 = Go[ap][bq], x10 = Go[bp][aq], x11 = Go[bp][bq];
      const cplx e01 = cmul(eq, x01), e11 = cmul(eq, x11);
      const cplx y00 = make_double2(cq * x00.x - sq * e01.x, cq * x00.y - sq * e01.y);
      const cplx y01 = make_double2(sq * x00.x + cq * e01.x, sq * x00.y + cq * e01.y);
      const cplx y10 = make_double2(cq * x10.x - sq * e11.x, cq * x10.y - sq * e11.y);
      const cplx y11 = make_double2(sq * x10.x + cq * e11.x, sq * x10.y + cq * e11.y);
      const cplx epc = cconj(ep);
      const cplx f10 = cmul(epc, y10), f11 = cmul(epc, y11);
      cplx z00 = make_double2(cp * y00.x - sp * f10.x, cp * y00.y - sp * f10.y);
      cplx z01 = make_double2(cp * y01.x - sp * f11.x, cp * y01.y - sp * f11.y);
      cplx z10 = make_double2(sp * y00.x + cp * f10.x, sp * y00.y + cp * f10.y);
      cplx z11 = make_double2(sp * y01.x + cp * f11.x, sp * y01.y + cp * f11.y);
      if (pr == qc) { z00.y = 0.0; z11.y = 0.0; }   // diagonal of a Hermitian matrix
      Gn[ap][aq] = z00; Gn[ap][bq] = z01; Gn[bp][aq] = z10; Gn[bp][bq] = z11;
      // W <- W R_q on this thread's 2x2 block (rows ap, bp)
      const cplx w00 = Ws[ap][aq], w01 = Ws[ap][bq], w10 = Ws[bp][aq], w11 = Ws[bp][bq];
      const cplx g01 = cmul(eq, w01), g11 = cmul(eq, w11);
      Ws[ap][aq] = make_double2(cq * w00.x - sq * g01.x, cq * w00.y - sq * g01.y);
      Ws[ap][bq] = make_double2(sq * w00.x + cq * g01.x, sq * w00.y + cq * g01.y);
      Ws[bp][aq] = make_double2(cq * w10.x - sq * g11.x, cq * w10.y - sq * g11.y);
      Ws[bp][bq] = make_double2(sq * w10.x + cq * g11.x, sq * w10.y + cq * g11.y);
      cur ^= 1;
      __syncthreads();
    }
    my_off2 = warp_max(my_off2);
    if (lane == 0) sh_red[w] = my_off2;
    __syncthreads();
    double so = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) so = fmax(so, sh_red[k]);
    __syncthreads();
    if (so < inner_tol * inner_tol) break;
  }
  if (cur) {                                      // final G lives in G2: the sort below reads Gs diagonals
    if (t < PR) Gs[t][t] = G2[t][t];
    __syncthreads();
  }
  // sort eigenvalues descending: perm[rank] = index  (identity first, so that non-finite input can never index out of bounds)
  if (t < PR) perm[t] = t;
  __syncthreads();
  if (t < PR) {
    const double li = Gs[t][t].x;
    int rank = 0;
    for (int j = 0; j < PR; ++j) {
      const double lj = Gs[j][j].x;
      rank += (lj > li) || (lj == li && j < t);
    }
    perm[rank] = t;
  }
  __syncthreads();
  // W^H planes with sorted columns: Aop[i][j] = conj(W[j][perm[i]])
  for (int e = t; e < PR * PR; e += 256) {
    const int i = e / PR, j = e % PR;
    const cplx v = Ws[j][perm[i]];
    Ps_re[i][j] = v.x;
    Ps_im[i][j] = -v.y;
  }
  __syncthreads();

  // ---------------- phase 3: P <- W^H P over all LD columns (DMMA), in place ----------------
  const int ntiles = ld / 8;
  for (int nt8 = w; nt8 < ntiles; nt8 += 8) {
    double br[4][2], bim[4][2], bn[4][2];
    const int col = nt8 * 8 + gq;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks)
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        const cplx x = Z[grow(ks * 8 + q + 4 * v) + col];
        br[ks][v] = x.x; bim[ks][v] = x.y; bn[ks][v] = -x.y;
      }
    double cr[2][4], ci[2][4];
#pragma unroll
    for (int m2 = 0; m2 < 2; ++m2) {
#pragma unroll
      for (int v = 0; v < 4; ++v) cr[m2][v] = ci[m2][v] = 0.0;
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        double ar[4], ai[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const int rr = m2 * 16 + gq + 8 * (v & 1), kk = ks * 8 + q + 4 * (v >> 1);
          ar[v] = Ps_re[rr][kk]; ai[v] = Ps_im[rr][kk];
        }
        dmma16x8x8(cr[m2], ar, br[ks]);
        dmma16x8x8(cr[m2], ai, bn[ks]);
        dmma16x8x8(ci[m2], ar, bim[ks]);
        dmma16x8x8(ci[m2], ai, br[ks]);
      }
    }
#pragma unroll
    for (int m2 = 0; m2 < 2; ++m2)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int rr = m2 * 16 + gq + 8 * (v >> 1);
        Z[grow(rr) + nt8 * 8 + 2 * q + (v & 1)] = cmake(cr[m2][v], ci[m2][v]);
      }
  }
}

// ------------------------------------------------------------------------------------------------
// one CTA per chain: row norms -> singular values, rank sort, write U_k S_k and V_k^H, update slots
__global__ void __launch_bounds__(1024) svd_extract_kernel(cplx* __restrict__ base, long long chain_stride, double* __restrict__ slots,
                                                           int n_slots, long long Z_, long long US_, long long Vh_, SvdGeom g,
                                                           int keep, int nr_bulk, int slot_lognorm, int slot_trunc, const int* __restrict__ mask,
                                                           int mask_want) {
  if (mask && mask[blockIdx.x] != mask_want) return;
  extern __shared__ double dyn[];
  double* s2 = dyn;                                   // p_pad
  int* idx = reinterpret_cast<int*>(dyn + g.p_pad);   // keep
  __shared__ double red[34];
  cplx* cb = base + (long long)blockIdx.x * chain_stride;
  const cplx* Z = cb + Z_;
  cplx* US = cb + US_;
  cplx* Vh = cb + Vh_;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5, nw = blockDim.x >> 5;
  for (int i = w; i < g.p_pad; i += nw) {
    double acc = 0.0;
    const cplx* row = Z + (long long)i * g.ld;
    for (int c = lane; c < g.q_pad; c += 32) acc += cabs2(row[c]);
    acc = warp_sum(acc);
    if (lane == 0) s2[i] = (acc == acc && acc < 1e300) ? acc : 0.0;   // non-finite rows are reported by the NaN guard op, not by a fault here
  }
  for (int k = t; k < keep; k += blockDim.x) idx[k] = 0;
  __syncthreads();
  double part = 0.0;
  for (int i = t; i < g.p_pad; i += blockDim.x) part += s2[i];
  const double total = block_sum(part, red);
  double disc_part = 0.0;
  for (int i = t; i < g.p_pad; i += blockDim.x) {
    const double si = s2[i];
    int rank = 0;
    for (int j = 0; j < g.p_pad; ++j) {
      const double sj = s2[j];
      rank += (sj > si) || (sj == si && j < i);
    }
    if (rank < keep) idx[rank] = i;
    else disc_part += si;                    // summed directly: total - kept would cancel
  }
  __syncthreads();
  const double disc = block_sum(disc_part, red);
  const double frob = sqrt(total);
  const double scale = (nr_bulk && frob > 0.0) ? 1.0 / frob : 1.0;
  const int m = g.m, n = g.n;
  if (g.mode_t) {
    // A = Yhat^T diag(s) conj(J):  US[r][k] = Y[idx_k][r] * scale ;  Vh[k][c] = conj(J[idx_k][c])
    for (long long e = t; e < (long long)m * keep; e += blockDim.x) {
      const int r = (int)(e / keep), k = (int)(e % keep);
      US[e] = cscale(Z[(long long)idx[k] * g.ld + r], scale);
    }
    for (long long e = t; e < (long long)keep * n; e += blockDim.x) {
      const int k = (int)(e / n), c = (int)(e % n);
      Vh[e] = cconj(Z[(long long)idx[k] * g.ld + g.q_pad + c]);
    }
  } else {
    // A = J^H diag(s) Yhat:  US[r][k] = conj(J[idx_k][r]) s_k scale ;  Vh[k][c] = Y[idx_k][c] / s_k
    for (long long e = t; e < (long long)m * keep; e += blockDim.x) {
      const int r = (int)(e / keep), k = (int)(e % keep);
      US[e] = cscale(cconj(Z[(long long)idx[k] * g.ld + g.q_pad + r]), sqrt(s2[idx[k]]) * scale);
    }
    for (long long e = t; e < (long long)keep * n; e += blockDim.x) {
      const int k = (int)(e / n), c = (int)(e % n);
      const double sk = sqrt(s2[idx[k]]);
      Vh[e] = sk > 0.0 ? cscale(Z[(long long)idx[k] * g.ld + c], 1.0 / sk) : cmake(0.0, 0.0);
    }
  }
  if (t == 0) {
    double* sl = slots + (long long)blockIdx.x * n_slots;
    if (nr_bulk && slot_lognorm >= 0 && frob > 0.0) sl[slot_lognorm] += log(frob);
    if (slot_trunc >= 0 && total > 0.0) sl[slot_trunc] += sqrt(disc / total);
  }
}

__global__ void svd_fro_kernel(const cplx* __restrict__ base, long long chain_stride, long long A_, long long n, double* __restrict__ fro2) {
  __shared__ double red[34];
  const cplx* A = base + (long long)blockIdx.x * chain_stride + A_;
  double acc = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) acc += cabs2(A[i]);
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) fro2[blockIdx.x] = acc;
}

__global__ void fill_kernel(double* p, int n, double v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ------------------------------------------------------------------------------------------------
// Sweep control on the device (one thread each).  begin: which chains take part (off_prev = huge), zero the sweep counter.
// end of a sweep: this sweep's measure becomes the next one's "previous"; another sweep iff some chain is above tolerance and
// the budget is not spent; a chain that runs out of budget is reported in the engine's status slot (include/kbp.h).
__global__ void svd_exact_begin_kernel(SvdCtl* __restrict__ ctl, const int* __restrict__ mask, int mask_want, double* __restrict__ off_prev, int nb,
                                       cudaGraphConditionalHandle h_sweep, int use_handle) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  int any = 0;
  for (int c = 0; c < nb; ++c) {
    const bool on = !mask || mask[c] == mask_want;
    off_prev[c] = on ? 1e300 : 0.0;
    if (on) { any = 1; ctl->counters[4] += 1; }
  }
  ctl->sweeps = 0;
  ctl->any_sweep = any;
  if (use_handle) cudaGraphSetConditional(h_sweep, any ? 1u : 0u);
}

__global__ void svd_exact_sweep_end_kernel(SvdCtl* __restrict__ ctl, double* __restrict__ off_prev, const double* __restrict__ off_cur, int nb,
                                           double tol, int max_sweeps, double* __restrict__ slots, int n_slots,
                                           cudaGraphConditionalHandle h_sweep, int use_handle) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int s = ctl->sweeps + 1;
  int any = 0;
  for (int c = 0; c < nb; ++c) {
    if (!(off_prev[c] >= tol)) continue;                     // took no part in this sweep
    double v = off_cur[c];
    if (!(v == v)) v = 0.0;                                   // non-finite input: reported by the program's NaN guard op
    if (v >= tol && s >= max_sweeps) {
      slots[(long long)c * n_slots + n_slots - 1] += 1.0;
      ctl->counters[7] += 1;
      v = 0.0;
    }
    off_prev[c] = v;
    any |= v >= tol;
  }
  ctl->sweeps = s;
  ctl->counters[6] += 1;
  ctl->any_sweep = any;
  if (use_handle) cudaGraphSetConditional(h_sweep, any ? 1u : 0u);
}

static void svd_exact_sweep(const Arena& a, int64_t work, const SvdGeom& g, double* prev, double* cur, double* fro2, cudaGraphConditionalHandle h_sweep) {
  cudaMemsetAsync(cur, 0, sizeof(double) * a.nb, a.stream);
  for (int r = 0; r < g.nblk - 1; ++r) {
    svd_round_kernel<<<dim3(g.nblk / 2, a.nb), 256, SVD_ROUND_SMEM, a.stream>>>(a.base, a.chain_stride, work, g, r, SVD_TOL, prev, cur, fro2, SVD_INNER_LO, a.ctl);
    ++*a.launches;
  }
  svd_exact_sweep_end_kernel<<<1, 32, 0, a.stream>>>(a.ctl, prev, cur, a.nb, SVD_TOL, SVD_MAX_SWEEPS, a.slots, a.n_slots, h_sweep, a.capture ? 1 : 0);
  ++*a.launches;
}

// Exact path: block one-sided Jacobi on the chains selected by a.mask (all if null).  The sweep loop is a WHILE node in
// graph mode and a host loop over the device's control block otherwise.  Returns sweeps (host mode) or 1, < 0 on CUDA failure.
int svd_exact(const Arena& a, int64_t A, int64_t US, int64_t Vh, int64_t work, int64_t m, int64_t n, int64_t keep, int nr_bulk,
              int slot_lognorm, int slot_trunc) {
  static const bool debug = getenv("KBP_SVD_DEBUG") != nullptr;
  if (debug) fprintf(stderr, "[kbp svd %lldx%lld keep %lld] block-Jacobi path\n", (long long)m, (long long)n, (long long)keep);
  SvdGeom g = svd_geom(m, n);
  {
    long long total = (long long)g.p_pad * g.ld;
    int gx = (int)((total + 255) / 256);
    if (gx > 148 * 8) gx = 148 * 8;
    svd_init_kernel<<<dim3(gx, a.nb), 256, 0, a.stream>>>(a.base, a.chain_stride, A, work, g, a.mask, a.mask_want);
    ++*a.launches;
  }
  // flags of the exact path live behind those of the subspace iteration (both may be in flight for different chains)
  double* base = a.svd_off + (6 + TSVD_NPART * TSVD_PART_STRIDE) * (size_t)a.nb;
  double* prev = base;
  double* cur = base + a.nb;
  double* fro2 = base + 2 * a.nb;
  svd_fro_kernel<<<a.nb, 512, 0, a.stream>>>(a.base, a.chain_stride, A, m * n, fro2);
  ++*a.launches;
  const cudaGraphConditionalHandle h_sweep = new_cond_handle(a);
  svd_exact_begin_kernel<<<1, 32, 0, a.stream>>>(a.ctl, a.mask, a.mask_want, prev, a.nb, h_sweep, a.capture ? 1 : 0);
  ++*a.launches;
  int sweeps = 1;
  if (a.capture) {
    Arena body;
    if (!begin_cond_body(a, h_sweep, true, &body)) return -1;
    svd_exact_sweep(body, work, g, prev, cur, fro2, h_sweep);
    if (!end_body(body)) return -1;
  } else {
    sweeps = 0;
    while (true) {
      svd_exact_sweep(a, work, g, prev, cur, fro2, h_sweep);
      ++sweeps;
      cudaMemcpyAsync(a.ctl_host, a.ctl, sizeof(SvdCtl), cudaMemcpyDeviceToHost, a.stream);
      if (stream_wait(a) != cudaSuccess) return -1;
      if (!a.ctl_host->any_sweep) break;
    }
  }
  size_t dyn = sizeof(double) * g.p_pad + sizeof(int) * (size_t)keep + 16;
  svd_extract_kernel<<<a.nb, 1024, dyn, a.stream>>>(a.base, a.chain_stride, a.slots, a.n_slots, work, US, Vh, g, (int)keep, nr_bulk,
                                                     slot_lognorm, slot_trunc, a.mask, a.mask_want);
  ++*a.launches;
  phase_fix(a, Vh, US, m, n, keep, 1);
  return sweeps;
}

// A matrix with a short side p <= 128 that does not fit the in-shared-memory kernel as a whole (64 x 512 at D = 4): one
// Householder factorisation reduces it to p x p, which does.   wide:  A^H = Q R  ->  A = R^H Q^H,  R^H = US_s Vh_s,
// US = US_s, Vh = Vh_s Q^H;   tall:  A = Q R,  R = US_s Vh,  US = Q US_s.  Same singular values, same truncation.
static void svd_reduced(const Arena& a, int64_t A, int64_t US, int64_t Vh, int64_t work, int64_t m, int64_t n, int64_t keep, int nr_bulk,
                        int slot_lognorm, int slot_trunc) {
  const int64_t p = m < n ? m : n, q = m < n ? n : m;
  int64_t o = work;
  const int64_t T = o; o += round_up(q * p, 8);          // A^H (wide) / unused (tall)
  const int64_t Q = o; o += round_up(q * p, 8);
  const int64_t R = o; o += round_up(p * p, 8);
  const int64_t L = o; o += round_up(p * p, 8);
  const int64_t S = o; o += round_up(p * keep, 8);       // small factor that still has to be multiplied by Q
  const int64_t qw = o;                                  // QR workspace: q*p + q*p + p + 8
  if (m < n) {
    const int64_t dims[2] = {m, n}, perm[2] = {1, 0};
    permute(a, T, A, 1, 2, dims, perm);                  // A^H, n x m
    qr(a, T, Q, R, qw, n, m);
    const int64_t dr[2] = {m, m};
    permute(a, L, R, 1, 2, dr, perm);                    // R^H, m x m
    svd_small(a, L, m, US, S, m, m, keep, nr_bulk, slot_lognorm, slot_trunc);      // S = Vh_s (keep x m)
    gemm(a, Vh, S, Q, keep, n, m, OP_N, OP_C);           // Vh = Vh_s Q^H
  } else {
    qr(a, A, Q, R, qw, m, n);
    svd_small(a, R, n, S, Vh, n, n, keep, nr_bulk, slot_lognorm, slot_trunc);      // S = US_s (n x keep)
    gemm(a, US, Q, S, m, keep, n, OP_N, OP_N);           // US = Q US_s
  }
  phase_fix(a, Vh, US, m, n, keep, 1);
}

bool svd_reducible(int64_t m, int64_t n) {
  const int64_t p = m < n ? m : n;
  return p <= 128 && !svd_small_fits(m, n) && svd_small_fits(p, p);
}

// Dispatcher: in-smem Jacobi for small matrices, Householder reduction + in-smem Jacobi for short-and-wide ones, subspace
// iteration when only a small leading part is kept, block-Jacobi otherwise / as the exact path of the subspace iteration.
// host counters: [1] small, [8..] none; everything decided on the device is counted there (SvdCtl::counters).
int svd_truncate(const Arena& a, int64_t A, int64_t US, int64_t Vh, int64_t work, int64_t m, int64_t n, int64_t keep,
                 int nr_bulk, int slot_lognorm, int slot_trunc) {
  if (m == 0 || n == 0) return 0;
  if (svd_small_fits(m, n)) {
    svd_small(a, A, n, US, Vh, m, n, keep, nr_bulk, slot_lognorm, slot_trunc);
    phase_fix(a, Vh, US, m, n, keep, 1);
    ++a.counters[1];
    return 1;
  }
  if (svd_reducible(m, n)) {
    svd_reduced(a, A, US, Vh, work, m, n, keep, nr_bulk, slot_lognorm, slot_trunc);
    ++a.counters[0];
    return 1;
  }
  const int b = tsvd_block(m, n, keep);
  if (b > 0) return svd_truncate_subspace(a, A, US, Vh, work, m, n, keep, nr_bulk, slot_lognorm, slot_trunc, b);
  Arena all = a;
  all.mask = nullptr;
  return svd_exact(all, A, US, Vh, work, m, n, keep, nr_bulk, slot_lognorm, slot_trunc);
}

void init_svd_attributes() {
  cudaFuncSetAttribute(svd_round_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SVD_ROUND_SMEM);
}

}  // namespace kbp
