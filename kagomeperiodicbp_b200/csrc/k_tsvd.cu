// Rank-`keep` truncated SVD of a LARGE complex128 matrix by block subspace iteration -- the truncation
// mps.right_canonical asks for (src/libs/bmpslib.py:733-772) keeps chi = 2 D^2 of chi D^2 singular triplets,
// so the full factorisation numpy computes there is ~10x more work than the answer needs.
//
//   Q0 (n x b) pseudo-random, b = 2.5 keep                             [deterministic hash, no RNG state]
//   repeat:  W = A Q ;  Y = orth(W) ;  Z = A^H Y ;  Q = orth(Z)        [DMMA ZGEMMs + Cholesky-QR]
//   Rayleigh-Ritz:  W = A Q = Y R  (Cholesky-QR twice, R = R2 R1, b x b),  R = Ur S Vb^H  by the in-smem
//   Jacobi kernel (k_svd_small.cu) ->  Vh = Vb_k^H Q^H  (keep x n, orthonormal rows),  US = A Vh^H.
//   accept iff  max_j || (I - Vh^H Vh) A^H US_j || / (s_j s_1)  <=  TSVD_RES_TOL  and  s_keep / s_1 >= TSVD_MIN_RATIO;
//   otherwise iterate further, and after TSVD_MAX_ITERS fall back to the full block-Jacobi
//   SVD (k_svd.cu).  The Ritz vectors j <= keep converge like (s_{b+1} / s_j)^(2 it): the boundary-MPS spectra of
//   the Kagome block have s_{3 chi} / s_chi ~ 0.05..0.15, i.e. 4-8 iterations for a 1e-13 residual.
//
// What is returned is an orthonormal basis Vh of the dominant right singular subspace and US = A Vh^H, so
// US Vh is exactly the projection of A on that subspace: the same truncated state the reference keeps, in a
// different (irrelevant) gauge of the kept bond.  The discarded weight is measured directly as
// ||A - US Vh||_F^2, not as a difference of large numbers.
#include "kbp_common.cuh"
#include "kbp_ops.cuh"

#include <mutex>
#include <vector>

#include <math.h>
#include <stdio.h>
#include <stdlib.h>

namespace kbp {

// ---- developer aid (KBP_TSVD_PROF=1, with KBP_GRAPHS=0): in-situ time of each kernel category of the subspace-iteration
// SVD, measured with events on the chain's own stream; totals over all chains are printed when the process exits.
namespace {
struct CatProf {
  bool on = getenv("KBP_TSVD_PROF") != nullptr;
  std::vector<cudaEvent_t> pool;
  std::vector<int> cats;
  size_t used = 0;
  void mark(cudaStream_t st, int cat) {
    if (!on) return;
    if (used == pool.size()) { cudaEvent_t e; cudaEventCreate(&e); pool.push_back(e); }
    cudaEventRecord(pool[used++], st);
    cats.push_back(cat);
  }
  void flush();
};
const char* const CAT_NAMES[8] = {"gemm A Q / A^H W", "gram gemm", "chol", "trsm", "small svd", "rayleigh-ritz gemms + phase", "checks + misc", "start"};
std::mutex g_prof_mu;
double g_prof_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
long long g_prof_n[8] = {0, 0, 0, 0, 0, 0, 0, 0};
void CatProf::flush() {
  if (!on || used < 2) { used = 0; cats.clear(); return; }
  std::lock_guard<std::mutex> lk(g_prof_mu);
  static bool registered = false;
  if (!registered) {
    registered = true;
    atexit([] {
      double tot = 0;
      for (int c = 0; c < 8; ++c) tot += g_prof_ms[c];
      for (int c = 0; c < 7; ++c)
        fprintf(stderr, "[kbp tsvd prof] %-28s %9.2f ms  %5.1f %%  (%lld spans, %.1f us each)\n", CAT_NAMES[c], g_prof_ms[c], 100.0 * g_prof_ms[c] / (tot > 0 ? tot : 1),
                g_prof_n[c], g_prof_n[c] ? 1e3 * g_prof_ms[c] / g_prof_n[c] : 0.0);
    });
  }
  for (size_t k = 1; k < used; ++k) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, pool[k - 1], pool[k]) == cudaSuccess) { g_prof_ms[cats[k]] += ms; ++g_prof_n[cats[k]]; }
  }
  used = 0;
  cats.clear();
}
thread_local CatProf t_prof;
}  // namespace
#define PM(cat) t_prof.mark(a.stream, cat)


constexpr int TSVD_BMAX = 112;            // widest block whose b x b Cholesky fits one CTA's shared memory
constexpr int TSVD_BMAX2 = 192;           // widest block at all: two column blocks orthogonalised by block Gram-Schmidt (D = 6:
                                          // keep 72 / 82 -> b = 184 / 192), Rayleigh-Ritz SVD on the cluster Jacobi kernel
constexpr int TSVD_B1 = 96;               // first column block of a wide panel
constexpr double TSVD_RES_TOL = 2e-13;
constexpr double TSVD_PIVOT_DEAD = 1e-13;  // pivot / diagonal below this: the column is numerically dependent -> dropped
// Dropped directions carry at most ~3e-7 of a column's norm (pivot ratio 1e-13), i.e. singular values below 3e-7 s_1.
// They can only belong to the kept triplets when the spectrum collapses inside the kept part, so a block whose keep-th
// Ritz value is below this fraction of the first (pivot ratio 1e-12: 10x above the drop threshold) goes to the exact path.
constexpr double TSVD_MIN_RATIO = 1e-6;

static inline int64_t rup8(int64_t x) { return (x + 7) / 8 * 8; }

// block = 2.0 x keep.  Measured on the D=4, N=3 side program (B200, whole program as one graph, profiles/r02_SUMMARY.md):
// 1.5 -> 136 ms, 1.7 -> 122, 2.0 -> 112.5, 2.2 -> 132, 2.5 -> 133, 3.0 -> 151 per chain: a wider block saves iterations
// (8.0 at 2.5 vs 9.6 at 2.0 on average) but every b x b kernel of an iteration (Cholesky, Jacobi, triangular solve) gets slower
constexpr int TSVD_BLOCK_FACTOR = 2;

int tsvd_block(int64_t m, int64_t n, int64_t keep) {
  const int64_t p = m < n ? m : n;
  int64_t b = rup8(TSVD_BLOCK_FACTOR * keep);
  if (b > TSVD_BMAX2) b = TSVD_BMAX2;
  if (b < keep + 8 || b * 100 > p * 80) return 0;     // not worth it / not applicable
  return (int)b;
}

int64_t tsvd_work_elems(int64_t m, int64_t n) {
  const int64_t q = m < n ? n : m, b = TSVD_BMAX2;
  return 6 * rup8(q) * b + 17 * b * b + m * n + 64;
}

// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long splitmix(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__global__ void tsvd_randq_kernel(cplx* __restrict__ base, long long chain_stride, long long Q_, long long total) {
  cplx* Q = base + (long long)blockIdx.y * chain_stride + Q_;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const unsigned long long h = splitmix((unsigned long long)e * 2 + 12345), h2 = splitmix(h);
    Q[e] = cmake((double)(h >> 11) * (1.0 / 9007199254740992.0) - 0.5, (double)(h2 >> 11) * (1.0 / 9007199254740992.0) - 0.5);
  }
}

// ------------------------------------------------------------------------------------------------
// One CTA per chain: Cholesky G = R^H R of a b x b Hermitian Gram matrix (given as `nsplit` partial sums) in shared
// memory, blocked by panels of 16:
//   A  the diagonal block is factored by 8 warps, one thread per entry kept in a register; the pivot row / column of each
//      of the 16 dependent steps goes through a double-buffered shared-memory line and ONE 256-thread named barrier
//      (a single warp doing this alone is ~5x slower: nothing hides its dependent-issue latency);
//   B  the panel rows by forward substitution, one thread per column, the column in registers;
//   C  the trailing update, block-parallel.
// R^{-1} is never formed: the orthonormalised block Y R^{-1} is a triangular solve per row (trsm_kernel), which is both
// cheaper than inverting in one CTA and more accurate.  Columns whose pivot is below TSVD_PIVOT_DEAD of their diagonal are
// dropped (row of R = 0, dinv = 0: the orthonormalised block gets a zero column there).  stat[chain] = min over live
// columns of pivot/diagonal.  Outputs: R (b x b, upper, row-major), Dinv (b entries, 1/R_jj in .x).
constexpr int CNB = 16;

struct CholWork {
  cplx* S;          // b x ld, upper triangle = Gram matrix in, Cholesky factor R out
  double* diag0;    // [b] original diagonal
  double* dinv;     // [b] 1 / R_jj (0 for dropped columns)
  double* piv;      // [b] pivot of each column (-1: dropped)
  cplx* rowbuf;     // [4 * CNB] pivot row / column lines, double buffered
  int ld;
};

// Blocked Cholesky of the b x b Hermitian matrix in w.S (upper triangle read, R written in place), all threads of the CTA.
// Called with w.diag0 filled and the block synchronised.
__device__ __forceinline__ void chol_factor(const CholWork& w, int b, int t, int nt) {
  cplx* S = w.S;
  double* diag0 = w.diag0;
  double* dinv = w.dinv;
  double* piv = w.piv;
  cplx* rowbuf = w.rowbuf;
  const int ld = w.ld;
  for (int p0 = 0; p0 < b; p0 += CNB) {
    const int p1 = p0 + CNB < b ? p0 + CNB : b, pw = p1 - p0;
    // ---- phase A
    if (t < 256) {
      const int row = t >> 4, col = t & 15;
      const bool in = row < pw && col < pw;
      cplx v = in ? S[(p0 + row) * ld + p0 + col] : cmake(row == col ? 1.0 : 0.0, 0.0);
      if (col < row) v = cconj(in ? S[(p0 + col) * ld + p0 + row] : cmake(0.0, 0.0));   // Hermitian: fill the lower part
      for (int j = 0; j < CNB; ++j) {
        cplx* rb = rowbuf + (j & 1) * 2 * CNB;
        cplx* cbuf = rb + CNB;
        if (row == j) rb[col] = v;
        if (col == j) cbuf[row] = v;
        asm volatile("bar.sync 1, 256;");
        const double d = rb[j].x;
        const double d0 = j < pw ? diag0[p0 + j] : 1.0;
        const bool live = d0 > 0.0 && d > TSVD_PIVOT_DEAD * d0;      // NaN -> dropped
        const double ip = live ? rsqrt(d) : 0.0;
        if (t == 0 && j < pw) piv[p0 + j] = live ? d : -1.0;
        const cplx srj = cbuf[row], sju = rb[col];                   // S[row][j], S[j][col]
        const double ip2 = ip * ip;
        const double vx = (srj.x * sju.x - srj.y * sju.y) * ip2, vy = (srj.x * sju.y + srj.y * sju.x) * ip2;
        const bool below = row > j, right = col > j, mine = row == j;
        double nx = v.x, ny = v.y;
        nx = (below && right) ? nx - vx : nx;
        ny = (below && right) ? ((col == row) ? 0.0 : ny - vy) : ny;
        nx = (mine && right) ? nx * ip : nx;
        ny = (mine && right) ? ny * ip : ny;
        nx = (mine && col == j) ? (live ? d * ip : 0.0) : nx;
        ny = (mine && col == j) ? 0.0 : ny;
        v = cmake(nx, ny);
        if (t == 0 && j < pw) dinv[p0 + j] = ip;
      }
      if (in && col >= row) S[(p0 + row) * ld + p0 + col] = v;       // R (upper)
    }
    __syncthreads();
    const int rem = b - p1;
    if (rem > 0) {
      // ---- phase B: R[r][l] = (S[r][l] - sum_{r' < r} conj(R[r'][r]) R[r'][l]) / R[r][r],  l >= p1
      // right-looking forward substitution, 16 lanes per column l (lane r owns row r of the panel): in step k lane k's value is
      // final, goes to the other lanes by a half-warp shuffle, and every later row takes its term
      for (int cb0 = 0; cb0 < rem; cb0 += nt >> 4) {
        const int lc = cb0 + (t >> 4), r = t & 15;
        const bool valid = lc < rem && r < pw;
        const int l = p1 + (lc < rem ? lc : 0);
        cplx acc = valid ? S[(p0 + r) * ld + l] : cmake(0.0, 0.0);
        const double dv = r < pw ? dinv[p0 + r] : 0.0;
#pragma unroll
        for (int k = 0; k < CNB; ++k) {
          if (k < pw) {
            cplx x = cscale(acc, dv);
            x.x = __shfl_sync(0xffffffffu, x.x, k, 16);
            x.y = __shfl_sync(0xffffffffu, x.y, k, 16);
            if (r == k) acc = x;
            if (r > k && r < pw) {
              const cplx v = ccmul(S[(p0 + k) * ld + p0 + r], x);
              acc.x -= v.x; acc.y -= v.y;
            }
          }
        }
        if (valid) S[(p0 + r) * ld + l] = acc;
      }
      __syncthreads();
      // ---- phase C: trailing update  S[i][l] -= sum_{r in panel} conj(R[r][i]) R[r][l],  p1 <= i <= l
      // upper triangle only, folded into a (rem + 1) x ceil(rem / 2) rectangle: row rr carries matrix row rr (rem - rr entries)
      // followed by matrix row rem - 1 - rr (rr + 1 entries)
      for (int e = t; e < (rem + 1) * ((rem + 1) / 2); e += nt) {
        const int rr = e / (rem + 1), cc = e - rr * (rem + 1);
        int ii, ll;
        if (cc < rem - rr) { ii = rr; ll = rr + cc; }
        else { ii = rem - 1 - rr; ll = ii + (cc - (rem - rr)); }
        if (cc >= rem - rr && ii == rr) continue;                  // odd rem: the middle row is listed once
        const int i = p1 + ii, l = p1 + ll;
        cplx x = S[i * ld + l], x2 = cmake(0.0, 0.0);
        for (int r = p0; r + 1 < p1; r += 2) {
          const cplx v = ccmul(S[r * ld + i], S[r * ld + l]), v2 = ccmul(S[(r + 1) * ld + i], S[(r + 1) * ld + l]);
          x.x -= v.x; x.y -= v.y;
          x2.x -= v2.x; x2.y -= v2.y;
        }
        if (pw & 1) {
          const cplx v = ccmul(S[(p1 - 1) * ld + i], S[(p1 - 1) * ld + l]);
          x.x -= v.x; x.y -= v.y;
        }
        x.x += x2.x; x.y += x2.y;
        if (l == i) x.y = 0.0;
        S[i * ld + l] = x;
      }
      __syncthreads();
    }
  }
}

// The same factorisation, unblocked and REGISTER resident (b <= 32 NC, 512 threads): the upper triangle is dealt block-cyclically,
// thread (warp w, lane) holding the entries (i, c) with i = w + 16 r, c = lane + 32 k, so every pivot row belongs to ONE warp and
// the active part of the matrix stays spread over all 16 warps to the end.  A step is one barrier: the owner warp publishes the
// (unscaled) pivot row through a double-buffered shared-memory line, every thread reads the pivot, its rows' and its columns'
// entries of that line and applies the rank-1 update to its registers (rows already factored are skipped warp-uniformly).
// The blocked version above spends ~450 cycles per pivot step (three phases per panel, the trailing matrix through shared
// memory); here a step is one barrier + one line read + <= 6 complex FMAs per thread.  v[r][k] is used iff r <= 2 k + 1 (the
// other pairs lie below the diagonal for every lane; the compiler drops them).  R (upper) is left in w.S, as above.
constexpr int CREG_LINE = 128;                                     // entries of one pivot line (b <= 128)

// w.rowbuf: 4 * CREG_LINE entries (two double-buffered lines: the pivot row u_c and the multipliers a_c = conj(u_c) / pivot).
// The loop is software pipelined: in step j the warp that owns row j + 1 updates that row FIRST and publishes it for step
// j + 1 (pivot broadcast by shuffle -> 1 / pivot -> line stores) before it touches its other rows, so the chain
//     barrier -> line loads -> complex FMA of the next pivot row -> shuffle -> reciprocal -> line stores -> barrier
// is all that is serial; the other 15 warps' updates (<= 6 complex FMAs per thread) run beside it.  The update is branch-free
// inside a row: only the register block that crosses the diagonal (k == r / 2) is predicated per lane, blocks to the right of
// it are always inside the triangle, rows already factored are skipped per warp.  One SM's FP64 pipe (64 FMA / clk) bounds
// the kernel from below: b^3 / 3 complex MACs = 5.5 k cycles at b = 64, ~2x that with the triangle dealt as rectangles.
template <int NC>
struct CholReg {
  static constexpr int NR = 2 * NC;
  cplx (&v)[2 * NC][NC];
  const CholWork& w;
  const int b, lane, wp;
  double pd;                     // pivot of the row this warp published last
  bool plive;

  __device__ __forceinline__ CholReg(cplx (&v_)[2 * NC][NC], const CholWork& w_, int b_, int t) : v(v_), w(w_), b(b_), lane(t & 31), wp(t >> 5), pd(0.0), plive(false) {}

  // row register r of this warp -= a * (pivot line), a = conj(u_i) / pivot of the warp's row i = wp + 16 r
  __device__ __forceinline__ void update_row(int r, const cplx a, const cplx (&uc)[NC]) {
    const int i = wp + 16 * r, kd = r >> 1;
#pragma unroll
    for (int k = 0; k < NC; ++k) {
      if (k < kd) continue;
      if (k > kd || lane + 32 * k >= i) {
        v[r][k].x = fma(-a.x, uc[k].x, fma(a.y, uc[k].y, v[r][k].x));
        v[r][k].y = fma(-a.x, uc[k].y, fma(-a.y, uc[k].x, v[r][k].y));
      }
    }
  }

  // the warp that holds pivot row jn in row register rn puts it (and the multipliers) on line jn & 1
  __device__ __forceinline__ void publish(int rn, int jn) {
    const int kp = rn >> 1;
    cplx* rb = w.rowbuf + (jn & 1) * (2 * CREG_LINE);
    cplx* ra = rb + CREG_LINE;
    const double d = __shfl_sync(0xffffffffu, v[rn][kp].x, 16 * (rn & 1) + (jn & 15));
    const double d0 = w.diag0[jn];
    const bool live = d0 > 0.0 && d > TSVD_PIVOT_DEAD * d0;        // NaN -> dropped
    const double inv = live ? 1.0 / d : 0.0;
#pragma unroll
    for (int k = 0; k < NC; ++k) {
      if (k < kp) continue;
      rb[lane + 32 * k] = v[rn][k];
      ra[lane + 32 * k] = cmake(v[rn][k].x * inv, -v[rn][k].y * inv);
    }
    pd = d;
    plive = live;
  }

  __device__ __forceinline__ void run() {
    cplx* S = w.S;
    const int ld = w.ld;
    __syncthreads();                                               // w.diag0 complete
    if (wp == 0) publish(0, 0);
#pragma unroll
    for (int rj = 0; rj < NR; ++rj) {
      const int kp = rj >> 1;
      for (int jj = 0; jj < 16; ++jj) {
        const int j = rj * 16 + jj;
        if (j >= b) break;
        const cplx* rb = w.rowbuf + (j & 1) * (2 * CREG_LINE);
        const cplx* ra = rb + CREG_LINE;
        __syncthreads();
        cplx uc[NC], ai[NR];
#pragma unroll
        for (int k = 0; k < NC; ++k) uc[k] = k >= kp ? rb[lane + 32 * k] : cmake(0.0, 0.0);
#pragma unroll
        for (int r = 0; r < NR; ++r) ai[r] = r >= rj ? ra[wp + 16 * r] : cmake(0.0, 0.0);
        // the next pivot row first
        const bool next_here = jj < 15 ? wp == jj + 1 : wp == 0;   // warp-uniform
        if (j + 1 < b && next_here) {
          if (jj < 15) {
            update_row(rj, ai[rj], uc);
            publish(rj, j + 1);
          } else if (rj + 1 < NR) {
            update_row(rj + 1 < NR ? rj + 1 : rj, ai[rj + 1 < NR ? rj + 1 : rj], uc);
            publish(rj + 1 < NR ? rj + 1 : rj, j + 1);
          }
        }
        // the other rows below the pivot (rows >= b hold zeros)
#pragma unroll
        for (int r = 0; r < NR; ++r) {
          if (r < rj) continue;
          const bool below = r > rj || wp > jj;
          const bool done = (jj < 15 && r == rj && wp == jj + 1) || (jj == 15 && r == rj + 1 && wp == 0);
          if (below && !done) update_row(r, ai[r], uc);
        }
        if (wp == jj) {                                            // row j of R, off the critical path of the other warps
          const double ip = plive ? rsqrt(pd) : 0.0;
#pragma unroll
          for (int k = 0; k < NC; ++k) {
            if (k < kp) continue;
            const int c = lane + 32 * k;
            if (c > j && c < b) S[j * ld + c] = cscale(v[rj][k], ip);
            else if (c == j) S[j * ld + c] = cmake(plive ? pd * ip : 0.0, 0.0);
          }
          if (lane == 0) { w.piv[j] = plive ? pd : -1.0; w.dinv[j] = ip; }
        }
      }
    }
    __syncthreads();
  }
};

template <int NC>
__device__ __forceinline__ void chol_factor_reg(const CholWork& w, int b, int t, cplx (&v)[2 * NC][NC]) {
  CholReg<NC> c(v, w, b, t);
  c.run();
}

// inverses of the 16 x 16 diagonal blocks of R (what the blocked triangular solve multiplies by): X = R_pp^{-1}, one HALF WARP
// per column l of a block (lane i = row i): back substitution from row l upwards, the entry found in step k goes to the lanes
// above it by a shuffle, each adds its term.  16 short steps per column with all columns of all blocks in flight (the
// one-thread-per-column version before it was a 136-term dependent chain on 64 threads: as long as the factorisation).
// Xd: nblk x 16 x 16 (shared or global memory).
__device__ __forceinline__ void chol_diag_inverses(const CholWork& w, int b, cplx* __restrict__ Xd, int t, int nt) {
  const cplx* S = w.S;
  const int ld = w.ld;
  const int nblk = (b + CNB - 1) / CNB, units = nblk * CNB, per_pass = nt >> 4;
  const int hw = t >> 4, i = t & 15;
  for (int u0 = 0; u0 < units; u0 += per_pass) {                   // uniform trip count: every lane takes part in the shuffles
    const int u = u0 + hw;
    const bool valid = u < units;
    const int pb = valid ? u >> 4 : 0, l = u & 15, p0 = pb * CNB;
    const bool row_in = p0 + i < b;
    const double di = row_in ? w.dinv[p0 + i] : 0.0;
    cplx acc = cmake(0.0, 0.0), mine = cmake(0.0, 0.0);
#pragma unroll
    for (int k = CNB - 1; k >= 0; --k) {
      cplx xk = cmake(0.0, 0.0);
      if (i == k && k <= l) xk = k == l ? cmake(di, 0.0) : cscale(acc, -di);
      if (i == k) mine = xk;
      xk.x = __shfl_sync(0xffffffffu, xk.x, k, 16);
      xk.y = __shfl_sync(0xffffffffu, xk.y, k, 16);
      if (i < k && p0 + k < b && row_in) acc = cfma(S[(p0 + i) * ld + p0 + k], xk, acc);
    }
    if (valid) Xd[pb * CNB * CNB + i * CNB + l] = mine;
  }
}

// smallest pivot / diagonal over the live columns (first warp; the value is valid in lane 0)
__device__ __forceinline__ double chol_min_pivot(const CholWork& w, int b, int t) {
  double mn = 1.0;
  for (int i = t; i < b; i += 32)
    if (w.piv[i] > 0.0) mn = fmin(mn, w.piv[i] / w.diag0[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
  return mn;
}

// Gram matrix (sum of the split-K partials, upper triangle) straight into the registers of chol_factor_reg, then the factorisation
template <int NC>
__device__ __forceinline__ void chol_reg_from_partials(const CholWork& w, const cplx* __restrict__ G, int nsplit, int b, int t) {
  constexpr int NR = 2 * NC;
  const int lane = t & 31, wp = t >> 5;
  const long long bb = (long long)b * b;
  cplx v[NR][NC];
#pragma unroll
  for (int r = 0; r < NR; ++r)
#pragma unroll
    for (int k = 0; k < NC; ++k) {
      v[r][k] = cmake(0.0, 0.0);
      if (2 * k + 1 >= r) {
        const int i = wp + 16 * r, c = lane + 32 * k;
        if (i < b && c < b && c >= i) {
          const cplx* gp = G + (long long)i * b + c;
          cplx x = gp[0];
          if (nsplit == 4) {
            const cplx v1 = gp[bb], v2 = gp[2 * bb], v3 = gp[3 * bb];
            x = cadd(cadd(x, v1), cadd(v2, v3));
          } else {
            for (int sp = 1; sp < nsplit; ++sp) x = cadd(x, gp[(long long)sp * bb]);
          }
          v[r][k] = x;
          if (c == i) w.diag0[i] = x.x;
        }
      }
    }
  chol_factor_reg<NC>(w, b, t, v);
}

constexpr int CREG_BMAX = 96;             // widest matrix of the register-resident factorisation (NC = 3: 12 entries per thread)

// One kernel per register-block count NC (and one for the blocked fallback), so that each gets its own register
// allocation.  (Capping NC = 2 at 64 registers -- half an SM's register file, so that its CTA can start beside other work --
// was measured: 34 -> 40 us per launch and no gain with six program graphs in flight; the cap is off.)
struct CholArgs {
  long long G, R, Dinv, Xd;
  int nsplit, b;
  const int* mask;
  int mask_want;
  int ktime;
};

__device__ __forceinline__ void chol_kernel_tail(const CholWork& w, cplx* cb, const CholArgs& g, double* __restrict__ stat, int t, int nt) {
  const int b = g.b, ld = w.ld;
  const cplx* S = w.S;
  cplx* R = cb + g.R;
  for (int r = t >> 5; r < b; r += nt >> 5)
    for (int c = t & 31; c < b; c += 32) R[(long long)r * b + c] = c >= r ? S[r * ld + c] : cmake(0.0, 0.0);
  cplx* Dv = cb + g.Dinv;
  for (int i = t; i < b; i += nt) Dv[i] = cmake(w.dinv[i], 0.0);
  chol_diag_inverses(w, b, cb + g.Xd, t, nt);
  if (t < 32) {
    const double mn = chol_min_pivot(w, b, t);
    if (t == 0) stat[blockIdx.x] = fmin(stat[blockIdx.x], mn);
  }
}

__device__ __forceinline__ CholWork chol_work(unsigned char* raw, cplx* rowbuf, int b) {
  CholWork w;
  w.ld = b + 1;                                                    // odd row stride: the 16 rows of a panel fall into different banks
  w.S = reinterpret_cast<cplx*>(raw);
  w.diag0 = reinterpret_cast<double*>(w.S + (size_t)b * w.ld);
  w.dinv = w.diag0 + b;
  w.piv = w.dinv + b;
  w.rowbuf = rowbuf;
  return w;
}

// developer probe (KBP_KTIME=1): wall time of every Cholesky CTA by %globaltimer, summed on the device -- the same one-SM kernel
// timed alone and with other program graphs running beside it shows how much the neighbours' work on its SM costs it
__device__ unsigned long long g_ktime_ns = 0, g_ktime_n = 0;
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

template <int NC>
__global__ void __launch_bounds__(512, 1) chol_reg_kernel(cplx* __restrict__ base, long long chain_stride, CholArgs g, double* __restrict__ stat) {
  if (g.mask && g.mask[blockIdx.x] != g.mask_want) return;
  const unsigned long long kt0 = g.ktime ? globaltimer_ns() : 0ull;
  extern __shared__ __align__(16) unsigned char ch_raw[];
  __shared__ cplx rowbuf[4 * CREG_LINE];
  const CholWork w = chol_work(ch_raw, rowbuf, g.b);
  cplx* cb = base + (long long)blockIdx.x * chain_stride;
  const int t = threadIdx.x;
  chol_reg_from_partials<NC>(w, cb + g.G, g.nsplit, g.b, t);
  chol_kernel_tail(w, cb, g, stat, t, blockDim.x);
  if (g.ktime) {
    __syncthreads();
    if (t == 0) { atomicAdd(&g_ktime_ns, globaltimer_ns() - kt0); atomicAdd(&g_ktime_n, 1ull); }
  }
}

void gemm_ktime_report(const char* tag);

void ktime_report(const char* tag) {
  gemm_ktime_report(tag);
  unsigned long long ns = 0, n = 0;
  cudaMemcpyFromSymbol(&ns, g_ktime_ns, sizeof(ns));
  cudaMemcpyFromSymbol(&n, g_ktime_n, sizeof(n));
  if (n) fprintf(stderr, "[kbp ktime] %s: %llu Cholesky CTAs, %.2f us each (globaltimer, inside the kernel)\n", tag, n, 1e-3 * (double)ns / (double)n);
  ns = n = 0;
  cudaMemcpyToSymbol(g_ktime_ns, &ns, sizeof(ns));
  cudaMemcpyToSymbol(g_ktime_n, &n, sizeof(n));
}

__global__ void __launch_bounds__(512) chol_blocked_kernel(cplx* __restrict__ base, long long chain_stride, CholArgs g, double* __restrict__ stat) {
  if (g.mask && g.mask[blockIdx.x] != g.mask_want) return;
  extern __shared__ __align__(16) unsigned char ch_raw[];
  __shared__ cplx rowbuf[4 * CNB];
  const int b = g.b, nsplit = g.nsplit;
  const CholWork w = chol_work(ch_raw, rowbuf, b);
  cplx* S = w.S;
  const int ld = w.ld;
  cplx* cb = base + (long long)blockIdx.x * chain_stride;
  const cplx* G = cb + g.G;
  const int t = threadIdx.x, nt = blockDim.x;
  {
    // sum of the split-K partial Gram matrices; (row, column) from the warp / lane, no integer division, all partials of
    // several rows in flight at once
    const int lane = t & 31, wp = t >> 5, nw = nt >> 5;
    const long long bb = (long long)b * b;
    for (int r = wp; r < b; r += nw) {
      for (int c = lane; c < b; c += 32) {
        const cplx* gp = G + (long long)r * b + c;
        cplx v = gp[0];
        if (nsplit == 4) {
          const cplx v1 = gp[bb], v2 = gp[2 * bb], v3 = gp[3 * bb];
          v = cadd(cadd(v, v1), cadd(v2, v3));
        } else {
          for (int sp = 1; sp < nsplit; ++sp) v = cadd(v, gp[(long long)sp * bb]);
        }
        S[r * ld + c] = v;
      }
    }
    __syncthreads();
    for (int i = t; i < b; i += nt) w.diag0[i] = S[i * ld + i].x;
    __syncthreads();
    chol_factor(w, b, t, nt);
  }
  chol_kernel_tail(w, cb, g, stat, t, nt);
}

static void launch_chol(const Arena& a, int64_t Gp, int split, int64_t R_out, int64_t Dinv, int64_t Xd, int b, double* stat) {
  const size_t smem = sizeof(double2) * (size_t)b * (b + 1) + 3 * sizeof(double) * (size_t)b + 32;
  static const int ktime = getenv("KBP_KTIME") != nullptr;
  const CholArgs g{Gp, R_out, Dinv, Xd, split, b, a.mask, a.mask_want, ktime};
  if (b <= 32) chol_reg_kernel<1><<<a.nb, 512, smem, a.stream>>>(a.base, a.chain_stride, g, stat);
  else if (b <= 64) chol_reg_kernel<2><<<a.nb, 512, smem, a.stream>>>(a.base, a.chain_stride, g, stat);
  else if (b <= CREG_BMAX) chol_reg_kernel<3><<<a.nb, 512, smem, a.stream>>>(a.base, a.chain_stride, g, stat);
  else chol_blocked_kernel<<<a.nb, 512, smem, a.stream>>>(a.base, a.chain_stride, g, stat);
  ++*a.launches;
}

// Out (rows x b) = Y R^{-1} for upper-triangular R by block forward substitution over the 16-column panels:
//     x_p = (y_p - sum_{r < p} x_r R_{r,p}) X_pp,        X_pp = inverse of the diagonal block (from chol_kernel).
// One CTA per TRSM_ROWS rows, ONE WARP PER ROW: lane = (h, c), c = column inside the panel, h = which half of the two inner
// sums (over the solved entries, over the rows of X_pp) the lane adds up; the halves meet in one shuffle.  The kernel is a
// chain of dependent instructions per warp (~12 cycles each), so what counts is how few of them a warp executes: with one
// row per half warp and undivided sums the 64-column solve took ~1900 instructions per warp (15 us).
// The X_pp, the blocks of R above the diagonal and the solved entries live in shared memory.
constexpr int TRSM_ROWS = 16;

__global__ void __launch_bounds__(512, 2) trsm_kernel(cplx* __restrict__ base, long long chain_stride, long long Y_, long long R_, long long Xd_,
                                                   long long Out_, int rows, int b, const int* __restrict__ mask, int mask_want) {
  if (mask && mask[blockIdx.y] != mask_want) return;
  extern __shared__ __align__(16) unsigned char tr_raw[];
  const int nblk = (b + CNB - 1) / CNB;
  cplx* Xs = reinterpret_cast<cplx*>(tr_raw);                     // nblk x 16 x 16: inverses of the diagonal blocks
  cplx* xs = Xs + (size_t)nblk * CNB * CNB;                       // TRSM_ROWS x (16 nblk + 1): solved entries of the CTA's rows
  cplx* tmp = xs + TRSM_ROWS * (size_t)(nblk * CNB + 1);          // TRSM_ROWS x 17
  cplx* Rs = tmp + TRSM_ROWS * 17;                                // the blocks of R above the diagonal blocks, packed per block column
  cplx* cb = base + (long long)blockIdx.y * chain_stride;
  const cplx* R = cb + R_;
  const cplx* Xd = cb + Xd_;
  const int t = threadIdx.x;
  for (int e = t; e < nblk * CNB * CNB; e += blockDim.x) Xs[e] = Xd[e];
  // R is shared by every row: one coalesced pass through L2 instead of a dependent L2 load per inner-loop step
  // (block column pb holds rows [0, 16 pb) x columns [16 pb, 16 pb + 16) at offset 256 pb (pb - 1) / 2)
  for (int pb = 1; pb < nblk; ++pb) {
    cplx* dst = Rs + CNB * CNB * (pb * (pb - 1) / 2);
    for (int e = t; e < CNB * CNB * pb; e += blockDim.x) {
      const int i = e >> 4, col = pb * CNB + (e & 15);
      dst[e] = col < b ? __ldg(R + (long long)i * b + col) : cmake(0.0, 0.0);
    }
  }
  const int r = t >> 5, lane = t & 31, c = lane & 15, h = lane >> 4;
  const int row = blockIdx.x * TRSM_ROWS + r;
  const bool ok = row < rows;
  const cplx* y = cb + Y_ + (long long)row * b;
  cplx* out = cb + Out_ + (long long)row * b;
  cplx* xr = xs + r * (nblk * CNB + 1);
  cplx* tr = tmp + r * 17;
  // the row's entries, one per lane and pair of panels: issued before the barrier so their latency hides behind the staging
  cplx yv[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int col = (2 * u + h) * CNB + c;
    yv[u] = (ok && col < b) ? y[col] : cmake(0.0, 0.0);
  }
  __syncthreads();
  for (int pb = 0; pb < nblk; ++pb) {
    const int p0 = pb * CNB, col = p0 + c;
    // y[col] sits in lane (pb & 1, c), register pb >> 1 (panels >= 8: straight from memory)
    cplx acc;
    {
      const int u = pb >> 1;
      cplx mine = u == 0 ? yv[0] : u == 1 ? yv[1] : u == 2 ? yv[2] : u == 3 ? yv[3] : ((ok && col < b && h == (pb & 1)) ? y[col] : cmake(0.0, 0.0));
      if (h != (pb & 1)) mine = cmake(0.0, 0.0);
      acc = mine;                                                  // the half that does not hold y starts from zero
    }
    {
      const cplx* rc = Rs + CNB * CNB * (pb * (pb - 1) / 2) + c;  // column c of block column pb
      const int half = p0 >> 1, i0 = h * half, i1 = i0 + half;    // p0 is a multiple of 16: both halves have a multiple of 8 terms
      cplx a1 = cmake(0.0, 0.0), a2 = a1, a3 = a1;
      for (int i = i0; i < i1; i += 4) {                           // four independent chains
        const cplx v0 = cmul(xr[i], rc[i * CNB]), v1 = cmul(xr[i + 1], rc[(i + 1) * CNB]);
        const cplx v2 = cmul(xr[i + 2], rc[(i + 2) * CNB]), v3 = cmul(xr[i + 3], rc[(i + 3) * CNB]);
        acc.x -= v0.x; acc.y -= v0.y;
        a1.x -= v1.x; a1.y -= v1.y;
        a2.x -= v2.x; a2.y -= v2.y;
        a3.x -= v3.x; a3.y -= v3.y;
      }
      acc.x += (a1.x + a2.x) + a3.x; acc.y += (a1.y + a2.y) + a3.y;
    }
    acc.x += __shfl_xor_sync(0xffffffffu, acc.x, 16);
    acc.y += __shfl_xor_sync(0xffffffffu, acc.y, 16);
    if (h == 0) tr[c] = acc;
    __syncwarp();
    // x[c] = sum_{cp <= c} tr[cp] X[cp][c]: half h adds the rows cp in [8 h, 8 h + 8)
    cplx x = cmake(0.0, 0.0), x2 = x;
    const cplx* X = Xs + pb * CNB * CNB + (h * 8) * CNB + c;
    const cplx* trh = tr + h * 8;
#pragma unroll
    for (int cp = 0; cp < 8; cp += 2) {
      if (h * 8 + cp <= c) x = cfma(trh[cp], X[cp * CNB], x);
      if (h * 8 + cp + 1 <= c) x2 = cfma(trh[cp + 1], X[(cp + 1) * CNB], x2);
    }
    x.x += x2.x; x.y += x2.y;
    x.x += __shfl_xor_sync(0xffffffffu, x.x, 16);
    x.y += __shfl_xor_sync(0xffffffffu, x.y, 16);
    if (h == 0 && col < b) {
      xr[col] = x;
      if (ok) out[col] = x;
    }
    __syncwarp();
  }
}

// How far span(Vh) is from an invariant subspace of A^H A, and the discarded weight, in two launches.
//   C = US^H A (keep x n),  T = C Vh^H = US^H US (keep x keep, T_jj = s_j^2),  TV = T Vh,  P = US Vh (m x n)
//   stage 1 (grid NPART x nb): partial sums of  r_j = ||C_j - TV_j||^2  (rows j),  ||A||_F^2  and  ||A - P||_F^2
//   stage 2 (one CTA per chain): out[0] = max_j sqrt(r_j / (s_j^2 s_1^2)), out[1] = min_j s_j / s_1, out[2] = ||A - P||^2 / ||A||^2
// Only the part of the residual OUTSIDE span(Vh) counts (C - T Vh): the part inside is a change of gauge of the kept
// bond, and it is also where the rounding of US = A Vh^H (absolute error eps s_1, amplified by A^H to eps s_1^2) lands,
// which would otherwise put a floor of eps s_1 / s_j under the test.
constexpr int NPART = TSVD_NPART;              // enough CTAs to pull A and P (m x n each) through L2 at its bandwidth, not at one SM's latency
constexpr int PART_STRIDE = TSVD_PART_STRIDE;  // doubles per (chain, part): keep <= 128 row sums + 2 norms

__global__ void __launch_bounds__(256) tsvd_check1_kernel(const cplx* __restrict__ base, long long chain_stride, long long C_, long long TV_,
                                                          long long A_, long long P_, int m, int n, int keep, double* __restrict__ part,
                                                          const int* __restrict__ mask, int mask_want) {
  if (mask && mask[blockIdx.y] != mask_want) return;
  __shared__ double red[34];
  const cplx* cb = base + (long long)blockIdx.y * chain_stride;
  const cplx* C = cb + C_;
  const cplx* TV = cb + TV_;
  const cplx* A = cb + A_;
  const cplx* P = cb + P_;
  double* out = part + ((long long)blockIdx.y * NPART + blockIdx.x) * PART_STRIDE;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  // rows of C - TV: part x owns a column range
  const int c0 = (int)((long long)n * blockIdx.x / NPART), c1 = (int)((long long)n * (blockIdx.x + 1) / NPART);
  for (int j = w; j < keep; j += 8) {
    double acc = 0.0;
    for (int c = c0 + lane; c < c1; c += 32) {
      const cplx x = C[(long long)j * n + c], y = TV[(long long)j * n + c];
      const double dx = x.x - y.x, dy = x.y - y.y;
      acc += dx * dx + dy * dy;
    }
    acc = warp_sum(acc);
    if (lane == 0) out[j] = acc;
  }
  const long long mn = (long long)m * n;
  const long long e0 = mn * blockIdx.x / NPART, e1 = mn * (blockIdx.x + 1) / NPART;
  double fa = 0.0, fd = 0.0;
  for (long long e = e0 + t; e < e1; e += 256) {
    const cplx x = A[e], y = P[e];
    fa += cabs2(x);
    const double dx = x.x - y.x, dy = x.y - y.y;
    fd += dx * dx + dy * dy;
  }
  fa = block_sum(fa, red);
  fd = block_sum(fd, red);
  if (t == 0) { out[keep] = fa; out[keep + 1] = fd; }
}

__global__ void __launch_bounds__(128) tsvd_check2_kernel(const cplx* __restrict__ base, long long chain_stride, long long T_, int keep,
                                                          const double* __restrict__ part, double* __restrict__ resid, double* __restrict__ ratio,
                                                          double* __restrict__ discfrac, double* __restrict__ norms, const int* __restrict__ mask,
                                                          int mask_want) {
  if (mask && mask[blockIdx.x] != mask_want) return;
  __shared__ double s2[128], r2[128];
  __shared__ double sh[2];
  const cplx* T = base + (long long)blockIdx.x * chain_stride + T_;
  const double* pp = part + (long long)blockIdx.x * NPART * PART_STRIDE;
  const int t = threadIdx.x;
  if (t < keep) {
    double acc = 0.0;
    for (int x = 0; x < NPART; ++x) acc += pp[x * PART_STRIDE + t];
    r2[t] = acc;
    s2[t] = T[(long long)t * keep + t].x;
  }
  if (t < 2) {
    double acc = 0.0;
    for (int x = 0; x < NPART; ++x) acc += pp[x * PART_STRIDE + keep + t];
    sh[t] = acc;
  }
  __syncthreads();
  if (t == 0) {
    double smax = 0.0;
    for (int j = 0; j < keep; ++j) smax = fmax(smax, s2[j]);
    double worst = 0.0, smin = smax;
    for (int j = 0; j < keep; ++j) {
      if (s2[j] > 1e-30 * smax) worst = fmax(worst, sqrt(r2[j] / (s2[j] * smax)));
      smin = fmin(smin, s2[j]);
    }
    if (!(worst == worst)) worst = 1e300;
    resid[blockIdx.x] = worst;
    ratio[blockIdx.x] = (smax > 0.0 && smin > 0.0) ? sqrt(smin / smax) : 0.0;
    discfrac[blockIdx.x] = sh[0] > 0.0 ? sh[1] / sh[0] : 0.0;
    norms[2 * blockIdx.x] = sh[0];
    norms[2 * blockIdx.x + 1] = sh[1];
  }
}

// grid (FIN_CTAS, nb): scale US by 1 / ||A||_F (nr_bulk); CTA 0 of a chain updates the slots from the norms check2 left behind.
constexpr int FIN_CTAS = 8;
__global__ void __launch_bounds__(256) tsvd_finalize_kernel(cplx* __restrict__ base, long long chain_stride, double* __restrict__ slots, int n_slots,
                                                            long long US_, long long mk, int nr_bulk, int slot_lognorm, int slot_trunc,
                                                            const double* __restrict__ norms, const int* __restrict__ mask, int mask_want) {
  if (mask && mask[blockIdx.y] != mask_want) return;
  cplx* US = base + (long long)blockIdx.y * chain_stride + US_;
  const double fro2 = norms[2 * blockIdx.y], disc = norms[2 * blockIdx.y + 1];
  const double frob = sqrt(fro2);
  if (nr_bulk && frob > 0.0) {
    const double sc = 1.0 / frob;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < mk; e += (long long)gridDim.x * blockDim.x) US[e] = cscale(US[e], sc);
  }
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double* sl = slots + (long long)blockIdx.y * n_slots;
    if (nr_bulk && slot_lognorm >= 0 && frob > 0.0) sl[slot_lognorm] += log(frob);
    if (slot_trunc >= 0 && fro2 > 0.0) sl[slot_trunc] += sqrt(disc / fro2);
  }
}

// Canonical phase of the kept right singular vectors: row k of Vh (keep x n) is multiplied by conj(phase) of its
// largest-magnitude entry (first one on ties), so that entry becomes real positive; with us_too the column k of US
// (m x keep) gets the phase back, leaving US Vh unchanged.  This pins the gauge of the truncated bond: the sites of
// the next BP iteration are then continuous functions of the messages, which is what lets the subspace iteration be
// warm-started from the previous run's Ritz basis.  One CTA per chain, one warp per row.
__global__ void __launch_bounds__(1024) phase_fix_kernel(cplx* __restrict__ base, long long chain_stride, long long Vh_, long long US_, int m, int n,
                                                         int keep, int us_too, const int* __restrict__ mask, int mask_want) {
  if (mask && mask[blockIdx.x] != mask_want) return;
  cplx* Vh = base + (long long)blockIdx.x * chain_stride + Vh_;
  cplx* US = base + (long long)blockIdx.x * chain_stride + US_;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int k = w; k < keep; k += nw) {
    cplx* row = Vh + (long long)k * n;
    // phase reference: <r, row> real positive for a fixed pseudo-random vector r (continuous in the row, unlike "largest entry")
    cplx acc = cmake(0.0, 0.0);
    for (int c = lane; c < n; c += 32) {
      const unsigned long long h = splitmix(0x51ed27ull + (unsigned long long)c), h2 = splitmix(h);
      const cplx r = cmake((double)(h >> 11) * (1.0 / 9007199254740992.0) - 0.5, (double)(h2 >> 11) * (1.0 / 9007199254740992.0) - 0.5);
      acc = cadd(acc, ccmul(r, row[c]));
    }
    acc = warp_sum(acc);
    const double best = cabs2(acc);
    if (!(best > 0.0)) continue;
    const double inv = rsqrt(best);
    const cplx ph = cmake(acc.x * inv, acc.y * inv);
    __syncwarp();
    for (int c = lane; c < n; c += 32) {
      row[c] = cmulc(row[c], ph);                           // * conj(ph)
    }
    if (us_too)
      for (int r = lane; r < m; r += 32) US[(long long)r * keep + k] = cmul(US[(long long)r * keep + k], ph);
  }
}

void phase_fix(const Arena& a, int64_t Vh, int64_t US, int64_t m, int64_t n, int64_t keep, int us_too) {
  phase_fix_kernel<<<a.nb, 1024, 0, a.stream>>>(a.base, a.chain_stride, Vh, US, (int)m, (int)n, (int)keep, us_too, a.mask, a.mask_want);
  ++*a.launches;
}

__global__ void tsvd_fill_kernel(double* p, int n, double v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

void svd_small(const Arena& a, int64_t A, int64_t lda, int64_t US, int64_t Vh, int64_t m, int64_t n, int64_t keep, int nr_bulk,
               int slot_lognorm, int slot_trunc);

// dst (rows x w, contiguous) = src[:, c0 : c0 + w] of a rows x ld matrix
__global__ void tsvd_gather_cols_kernel(cplx* __restrict__ base, long long chain_stride, long long dst_, long long src_, int rows, int ld, int c0, int w,
                                        const int* __restrict__ mask, int mask_want) {
  if (mask && mask[blockIdx.y] != mask_want) return;
  cplx* cb = base + (long long)blockIdx.y * chain_stride;
  const long long total = (long long)rows * w;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / w;
    const int c = (int)(e - r * w);
    cb[dst_ + e] = cb[src_ + r * ld + c0 + c];
  }
}
// dst[:, c0 : c0 + w] (rows x ld) = src (rows x w, contiguous);  zero_rest: the other columns of those rows are zeroed
__global__ void tsvd_scatter_cols_kernel(cplx* __restrict__ base, long long chain_stride, long long dst_, long long src_, int rows, int ld, int c0, int w,
                                         const int* __restrict__ mask, int mask_want) {
  if (mask && mask[blockIdx.y] != mask_want) return;
  cplx* cb = base + (long long)blockIdx.y * chain_stride;
  const long long total = (long long)rows * w;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long r = e / w;
    const int c = (int)(e - r * w);
    cb[dst_ + r * ld + c0 + c] = cb[src_ + e];
  }
}
// x -= y  (n elements)
__global__ void tsvd_sub_kernel(cplx* __restrict__ base, long long chain_stride, long long x_, long long y_, long long n, const int* __restrict__ mask,
                                int mask_want) {
  if (mask && mask[blockIdx.y] != mask_want) return;
  cplx* cb = base + (long long)blockIdx.y * chain_stride;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) cb[x_ + e] = csub(cb[x_ + e], cb[y_ + e]);
}

static inline int grid1d(long long n) {
  long long g = (n + 255) / 256;
  return (int)(g > 148 * 8 ? 148 * 8 : (g < 1 ? 1 : g));
}

// Y (rows x b) <- Y Rinv with G = Y^H Y = R^H R.  `T` is a rows x b scratch; returns the buffer holding the result
// (Y and T swap roles).  R_out >= 0: also store R.  The Gram matrix is accumulated as GRAM_SPLIT partial sums over
// row ranges (more CTAs on a product whose output is only b x b) which the Cholesky kernel adds up.
constexpr int GRAM_SPLIT = 4;

static int64_t cholqr_pass_narrow(const Arena& a, int64_t Y, int64_t T, int64_t Gp, int64_t Dinv, int64_t R_out, int64_t rows, int b, double* stat) {
  const int split = rows >= 256 ? GRAM_SPLIT : 1;
  gemm_splitk(a, Gp, Y, Y, b, b, rows, OP_C, OP_N, split);
  PM(1);
  const int64_t Xd = Dinv + b;                                     // diagonal-block inverses behind the 1/diagonal entries
  launch_chol(a, Gp, split, R_out, Dinv, Xd, b, stat);
  PM(2);
  if (T >= 0) {                                                   // T < 0: only R is wanted
    const int nblk = (b + CNB - 1) / CNB;
    const size_t smem2 = sizeof(double2) * ((size_t)nblk * CNB * CNB + TRSM_ROWS * (size_t)(nblk * CNB + 1) + TRSM_ROWS * 17 +
                                            (size_t)CNB * CNB * (nblk * (nblk - 1) / 2)) + 32;
    trsm_kernel<<<dim3((unsigned)((rows + TRSM_ROWS - 1) / TRSM_ROWS), a.nb), 512, smem2, a.stream>>>(a.base, a.chain_stride, Y, R_out, Xd, T, (int)rows, b, a.mask,
                                                                                                      a.mask_want);
    ++*a.launches;
    PM(3);
  }
  return T;
}

// Wide panels (b > TSVD_BMAX): the b x b Cholesky no longer fits one CTA's shared memory.  The panel is split into two column
// blocks Y = [Y1 | Y2] (b1 = 96 columns, the rest) orthogonalised by block Gram-Schmidt with a Cholesky-QR per block:
//     Y1 = Q1 R11,   R12 = Q1^H Y2,   Y2 - Q1 R12 = Q2 R22        ->   Y = [Q1 | Q2] [[R11, R12], [0, R22]]
// (the callers repeat the pass on the last iteration, which makes it block classical Gram-Schmidt with reorthogonalisation).
// `X` = scratch of >= 2 * rows * b + 2 * b * b elements (panels 4 and 5 of the workspace).
static int64_t cholqr_pass(const Arena& a, int64_t Y, int64_t T, int64_t Gp, int64_t Dinv, int64_t R_out, int64_t rows, int b, double* stat, int64_t X = -1) {
  if (b <= TSVD_BMAX) return cholqr_pass_narrow(a, Y, T, Gp, Dinv, R_out, rows, b, stat);
  const int b1 = TSVD_B1, b2 = b - b1;
  const int64_t Y1 = X, Y2 = Y1 + rows * b1, Q1 = Y2 + rows * b2, Q2 = Q1 + rows * b1, R11 = Q2 + rows * b2, R22 = R11 + (int64_t)b1 * b1,
                R12 = R22 + (int64_t)b2 * b2, P2 = Y1;                        // Y1 is dead once Q1 exists: reused for Q1 R12
  const dim3 g1(grid1d(rows * b1), a.nb), g2(grid1d(rows * b2), a.nb);
  tsvd_gather_cols_kernel<<<g1, 256, 0, a.stream>>>(a.base, a.chain_stride, Y1, Y, (int)rows, b, 0, b1, a.mask, a.mask_want);
  tsvd_gather_cols_kernel<<<g2, 256, 0, a.stream>>>(a.base, a.chain_stride, Y2, Y, (int)rows, b, b1, b2, a.mask, a.mask_want);
  *a.launches += 2;
  cholqr_pass_narrow(a, Y1, Q1, Gp, Dinv, R11, rows, b1, stat);
  gemm(a, R12, Q1, Y2, b1, b2, rows, OP_C, OP_N);                           // R12 = Q1^H Y2
  gemm(a, P2, Q1, R12, rows, b2, b1, OP_N, OP_N);                           // Q1 R12
  tsvd_sub_kernel<<<g2, 256, 0, a.stream>>>(a.base, a.chain_stride, Y2, P2, rows * b2, a.mask, a.mask_want);
  ++*a.launches;
  cholqr_pass_narrow(a, Y2, Q2, Gp, Dinv, R22, rows, b2, stat);
  if (T >= 0) {
    tsvd_scatter_cols_kernel<<<g1, 256, 0, a.stream>>>(a.base, a.chain_stride, T, Q1, (int)rows, b, 0, b1, a.mask, a.mask_want);
    tsvd_scatter_cols_kernel<<<g2, 256, 0, a.stream>>>(a.base, a.chain_stride, T, Q2, (int)rows, b, b1, b2, a.mask, a.mask_want);
    *a.launches += 2;
  }
  if (R_out >= 0) {                                                          // assemble the b x b factor (rows b1.. of the left block are zero)
    zero(a, R_out, (int64_t)b * b);
    tsvd_scatter_cols_kernel<<<dim3(grid1d(b1 * b1), a.nb), 256, 0, a.stream>>>(a.base, a.chain_stride, R_out, R11, b1, b, 0, b1, a.mask, a.mask_want);
    tsvd_scatter_cols_kernel<<<dim3(grid1d(b1 * b2), a.nb), 256, 0, a.stream>>>(a.base, a.chain_stride, R_out, R12, b1, b, b1, b2, a.mask, a.mask_want);
    tsvd_scatter_cols_kernel<<<dim3(grid1d(b2 * b2), a.nb), 256, 0, a.stream>>>(a.base, a.chain_stride, R_out + (int64_t)b1 * b, R22, b2, b, b1, b2, a.mask,
                                                                               a.mask_want);
    *a.launches += 3;
  }
  return T;
}

// ------------------------------------------------------------------------------------------------
// Thin QR of a TALL matrix (m >= 4 n, 8 <= n <= 96) as Cholesky-QR twice:  A = Q1 R1,  Q1 = Q R2,  R = R2 R1  -- three
// launches per pass (split-K Gram product on the DMMA pipe, register Cholesky, triangular solve) instead of a Householder
// sweep whose every column costs two exchanges over distributed shared memory (512 x 32: ~190 us against ~60 us).
// Cholesky-QR squares the condition number, so it is used only where that is harmless: the pivots are invariant under
// column scaling, and the smallest pivot / diagonal of pass 1 bounds 1 / cond^2 of the column-scaled matrix.  With a ratio
// >= CHOLQR2_MIN_PIVOT the first pass leaves ||Q1^H Q1 - I|| <~ eps / ratio <= 1e-5 and the second pass brings it to eps.
// Anything else -- smaller pivots, numerically dependent (dropped) columns, non-finite entries -- is decided ON THE DEVICE, per
// chain, and redone by the Householder kernels, which are launched behind the decision with that per-chain predicate.
// The boundary-MPS sites of a converged BP run have scaled condition numbers of 1e2 .. 1e6 (measured on the op streams of
// the CPU tier); the rank-deficient sites of the first iterations from product messages take the fallback.
constexpr double CHOLQR2_MIN_PIVOT = 1e-11;

__global__ void cholqr2_decide_kernel(int* __restrict__ state, const double* __restrict__ stat, const cplx* __restrict__ base, long long chain_stride,
                                      long long R1_, long long R2_, int n) {
  // one warp per chain: lanes over the diagonal entries
  const int c = blockIdx.x;
  int bad = !(stat[c] >= CHOLQR2_MIN_PIVOT);                         // also NaN
  const cplx* R1 = base + (long long)c * chain_stride + R1_;
  const cplx* R2 = base + (long long)c * chain_stride + R2_;
  for (int j = threadIdx.x; j < n; j += 32)
    if (!(R1[(long long)j * n + j].x > 0.0) || !(R2[(long long)j * n + j].x > 0.0)) bad = 1;       // dropped column
  bad = __any_sync(0xffffffffu, bad);
  if (threadIdx.x == 0) state[c] = bad ? CHAIN_EXACT : CHAIN_ACCEPTED;
}

// ------------------------------------------------------------------------------------------------
// The decision after every Rayleigh-Ritz round, on the device (one thread): per chain accept / iterate further / exact path.
// A chain that is done leaves the RUNNING state, which is the per-chain predicate of every launch of the following rounds.
//   accept    residual <= TSVD_RES_TOL, Cholesky pivots of the round trustworthy, no collapse of the kept spectrum
//   exact     kept spectrum collapses with measurable discarded weight, non-finite flags, or the round budget is spent
constexpr double TSVD_PIVOT_TRUST = 1e-3;

__global__ void tsvd_decide_kernel(SvdCtl* __restrict__ ctl, int* __restrict__ state, double* __restrict__ stat, const double* __restrict__ resid,
                                   const double* __restrict__ ratio, const double* __restrict__ discf, int nb, int first, int max_rounds,
                                   int iters_first, int iters_more, cudaGraphConditionalHandle h_loop, cudaGraphConditionalHandle h_exact,
                                   int use_handles, const cplx* __restrict__ base, long long chain_stride, long long R1_, int b, int keep) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const int round = first ? 1 : ctl->round + 1;
  int any_run = 0, any_exact = 0;
  for (int c = 0; c < nb; ++c) {
    int st = first ? CHAIN_RUNNING : state[c];
    if (st == CHAIN_RUNNING) {
      const double pv = stat[c], rs = resid[c], ra = ratio[c], df = discf[c];
      const bool finite = pv == pv && rs == rs && ra == ra && df == df;
      const bool trusted = pv >= TSVD_PIVOT_TRUST;
      // A kept spectrum that spans more than six decades is only a problem if the block LOST directions of that size: the
      // Cholesky of the first iterations drops columns it cannot tell from rounding (< ~3e-7 of the leading direction), and
      // a dropped column stays zero.  If more than `keep` columns of the block are still alive in the Rayleigh-Ritz
      // factor, the block resolved a direction BELOW the kept ones, i.e. nothing of the kept size was dropped and the kept
      // set is the dominant one; the small kept directions themselves are as accurate as the large ones (the rounding of
      // A^H (A q_j) is relative to s_1 s_j: angle error ~ eps s_1 / s_j, contribution to the state ~ eps s_1).
      int live = 0;
      {
        const cplx* R1 = base + (long long)c * chain_stride + R1_;
        for (int j = 0; j < b; ++j) live += R1[(long long)j * b + j].x > 0.0;
      }
      const bool collapse = trusted && ra < TSVD_MIN_RATIO && df > 1e-24 && live <= keep;
      if (finite && trusted && !collapse && rs <= TSVD_RES_TOL) {
        st = CHAIN_ACCEPTED;
        ctl->counters[2] += 1;
        ctl->counters[5] += iters_first + (long long)(round - 1) * iters_more;
      } else if (!finite || collapse || round >= max_rounds) {
        st = CHAIN_EXACT;
        ctl->counters[3] += 1;
      }
    }
    state[c] = st;
    stat[c] = 1.0;                               // smallest Cholesky pivot ratio of the next round
    any_run |= st == CHAIN_RUNNING;
    any_exact |= st == CHAIN_EXACT;
  }
  ctl->round = round;
  ctl->any_run = any_run;
  ctl->any_exact = any_exact;
  if (use_handles) {
    cudaGraphSetConditional(h_loop, any_run ? 1u : 0u);
    cudaGraphSetConditional(h_exact, any_exact ? 1u : 0u);
  }
}

int svd_exact(const Arena& a, int64_t A, int64_t US, int64_t Vh, int64_t work, int64_t m, int64_t n, int64_t keep, int nr_bulk,
              int slot_lognorm, int slot_trunc);

// ---- conditional graph nodes ------------------------------------------------------------------------------------------
cudaGraphConditionalHandle new_cond_handle(const Arena& a) {
  cudaGraphConditionalHandle h = 0;
  if (a.capture) cudaGraphConditionalHandleCreate(&h, a.top_graph, 0, cudaGraphCondAssignDefault);
  return h;
}

bool begin_cond_body(const Arena& a, cudaGraphConditionalHandle h, bool is_while, Arena* body) {
  cudaStreamCaptureStatus st;
  unsigned long long id;
  cudaGraph_t g = nullptr;
  const cudaGraphNode_t* deps = nullptr;
  size_t nd = 0;
  if (a.depth >= 2) return false;
  if (cudaStreamGetCaptureInfo_v2(a.stream, &st, &id, &g, &deps, &nd) != cudaSuccess || st != cudaStreamCaptureStatusActive) return false;
  cudaGraphNodeParams p = {};
  p.type = cudaGraphNodeTypeConditional;
  p.conditional.handle = h;
  p.conditional.type = is_while ? cudaGraphCondTypeWhile : cudaGraphCondTypeIf;
  p.conditional.size = 1;
  cudaGraphNode_t node;
  if (cudaGraphAddNode(&node, g, deps, nd, &p) != cudaSuccess) return false;
  if (cudaStreamUpdateCaptureDependencies(a.stream, &node, 1, cudaStreamSetCaptureDependencies) != cudaSuccess) return false;
  *body = a;
  body->stream = a.body_stream[a.depth];
  body->depth = a.depth + 1;
  return cudaStreamBeginCaptureToGraph(body->stream, p.conditional.phGraph_out[0], nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
}

bool end_body(const Arena& body) {
  cudaGraph_t g = nullptr;
  return cudaStreamEndCapture(body.stream, &g) == cudaSuccess;
}

static cudaError_t read_ctl(const Arena& a) {
  cudaMemcpyAsync(a.ctl_host, a.ctl, sizeof(SvdCtl), cudaMemcpyDeviceToHost, a.stream);
  return stream_wait(a);
}

// ------------------------------------------------------------------------------------------------
// Workspace of one subspace truncation (complex128 elements from `work`)
struct TsvdBufs {
  int64_t panel[4];                  // four q x b panels
  int64_t Gp, Ri, Rs, R1, R2, Rm, Vbs, Tk, Pb;
  int64_t X;                         // scratch of the wide-panel Cholesky-QR (two panels + b x b)
};

// Rayleigh-Ritz on span(Q), the kept factors, and the two check kernels.  Q in panel `Qb`, `f0`, `f1` free panels.
static void rayleigh_ritz_and_check(const Arena& a, const TsvdBufs& w, int64_t A, int64_t US, int64_t Vh, int64_t m, int64_t n, int64_t keep,
                                    int b, int64_t Qb, int64_t f0, int64_t f1, bool single_pass) {
  double* stat = a.svd_off;
  double* resid = a.svd_off + a.nb;
  double* ratio = a.svd_off + 2 * a.nb;
  double* discf = a.svd_off + 3 * a.nb;
  double* norms = a.svd_off + 4 * a.nb;
  double* part = a.svd_off + 6 * a.nb;
  gemm(a, f0, A, Qb, m, b, n, OP_N, OP_N);                          // W = A Q -> f0
  PM(0);
  int64_t Rsmall;
  if (single_pass) {
    cholqr_pass(a, f0, -1, w.Gp, w.Ri, w.R1, m, b, stat, w.X);           // W = Y R1
    Rsmall = w.R1;
  } else {
    cholqr_pass(a, f0, f1, w.Gp, w.Ri, w.R1, m, b, stat, w.X);
    cholqr_pass(a, f1, -1, w.Gp, w.Ri, w.R2, m, b, stat, w.X);
    gemm(a, w.Rm, w.R2, w.R1, b, b, b, OP_N, OP_N);                 // W = Y (R2 R1)
    PM(5);
    Rsmall = w.Rm;
  }
  svd_small(a, Rsmall, b, -1, w.Vbs, b, b, b, 0, -1, -1);           // Vbs = Vb^H (b x b), rows by decreasing singular value
  PM(4);
  gemm(a, Vh, w.Vbs, Qb, keep, n, b, OP_N, OP_C);                   // Vh = Vb_k^H Q^H
  phase_fix(a, Vh, US, m, n, keep, 0);                              // canonical gauge of the kept bond
  gemm(a, US, A, Vh, m, keep, n, OP_N, OP_C);                       // US = A Vh^H
  gemm(a, f0, US, A, keep, n, m, OP_C, OP_N);                       // C = US^H A        -> f0
  gemm(a, w.Tk, f0, Vh, keep, keep, n, OP_N, OP_C);                 // T = C Vh^H
  gemm(a, f1, w.Tk, Vh, keep, n, keep, OP_N, OP_N);                 // TV = T Vh         -> f1
  gemm(a, w.Pb, US, Vh, m, n, keep, OP_N, OP_N);                    // P = US Vh
  PM(5);
  tsvd_check1_kernel<<<dim3(NPART, a.nb), 256, 0, a.stream>>>(a.base, a.chain_stride, f0, f1, A, w.Pb, (int)m, (int)n, (int)keep, part, a.mask, a.mask_want);
  tsvd_check2_kernel<<<a.nb, 128, 0, a.stream>>>(a.base, a.chain_stride, w.Tk, (int)keep, part, resid, ratio, discf, norms, a.mask, a.mask_want);
  *a.launches += 2;
  PM(6);
}

// One more round from the Ritz basis of the previous one: `TSVD_IT_MORE` FAST iterations (an odd number: Q ends in the panel
// it started in, so the round is a loop body with fixed buffer roles), Rayleigh-Ritz, check, decision.
constexpr int TSVD_IT_MORE = 3;

static void tsvd_more_round(const Arena& a, const TsvdBufs& w, int64_t A, int64_t US, int64_t Vh, int64_t m, int64_t n, int64_t keep, int b,
                            int64_t Qb, int64_t f0, int64_t f1, int64_t f2, int max_rounds, int iters_first,
                            cudaGraphConditionalHandle h_loop, cudaGraphConditionalHandle h_exact) {
  double* stat = a.svd_off;
  gemm(a, f2, Qb, w.Vbs, n, b, b, OP_N, OP_C);                      // Ritz vectors Q Vb, ordered         -> f2
  PM(5);
  int64_t cur = f2, other = Qb;
  for (int it = 0; it < TSVD_IT_MORE; ++it) {
    gemm(a, f0, A, cur, m, b, n, OP_N, OP_N);                       // W = A Q
    gemm(a, f1, A, f0, n, b, m, OP_C, OP_N);                        // Z = A^H W
    PM(0);
    cholqr_pass(a, f1, other, w.Gp, w.Ri, w.Rs, n, b, stat, w.X);        // Q = orth(Z) -> other
    const int64_t t = cur; cur = other; other = t;
  }
  // TSVD_IT_MORE odd: cur == Qb again
  rayleigh_ritz_and_check(a, w, A, US, Vh, m, n, keep, b, cur, f0, f1, true);
  tsvd_decide_kernel<<<1, 32, 0, a.stream>>>(a.ctl, a.chain_state, stat, a.svd_off + a.nb, a.svd_off + 2 * a.nb, a.svd_off + 3 * a.nb, a.nb, 0,
                                             max_rounds, iters_first, TSVD_IT_MORE, h_loop, h_exact, a.capture ? 1 : 0, a.base, a.chain_stride, w.R1, b, (int)keep);
  ++*a.launches;
}

// Iterations of round 1 from the pseudo-random block (the spectra of the Kagome block need 4-8 for a 1e-13 residual, see the top).
constexpr int TSVD_IT_COLD = 7;
// cold start: after TSVD_SAFE_ITERS SAFE iterations the block is already ordered well enough (contamination of column j by a
// larger direction i has decayed as (s_j/s_i)^(2k), one fast step amplifies it by (s_i/s_j)^2) for the FAST form
constexpr int TSVD_SAFE_ITERS = 2;

// Two kinds of iteration.  SAFE (cold start, Q arbitrary): W = A Q, Y = orth(W), Z = A^H Y, Q = orth(Z).  FAST (Q holds
// approximate Ritz vectors in decreasing order -- after TSVD_SAFE_ITERS SAFE iterations of a cold start, or after a Rayleigh-Ritz
// step): the columns of A Q and of A^H A Q are then nearly orthogonal, their Gram matrices are diagonally dominant after
// scaling, and ONE Cholesky-QR of Z = A^H (A Q) per iteration is as accurate as the safe sequence (the Cholesky kernel
// reports its smallest pivot / diagonal; a round built on a pivot ratio below TSVD_PIVOT_TRUST is not accepted).
//
// No host decision anywhere: round 1 is a fixed launch sequence, every further round is the body of a WHILE node (graph
// mode) or of a host loop reading the device's control block (host-driven mode), the exact path is an IF node.
// Returns the number of launches-visible rounds (>= 1), < 0 on a CUDA failure.
int svd_truncate_subspace(const Arena& a0, int64_t A, int64_t US, int64_t Vh, int64_t work, int64_t m, int64_t n, int64_t keep,
                          int nr_bulk, int slot_lognorm, int slot_trunc, int b) {
  static const bool debug = getenv("KBP_SVD_DEBUG") != nullptr;
  // An op that needed r > 1 rounds when its program ran host-driven (previous BP iteration: nearly the same spectrum) gets
  // the iterations of those rounds up front in the captured graph: one Rayleigh-Ritz step + check instead of r.
  int it_cold = TSVD_IT_COLD;
  if (a0.capture && a0.tsvd_rounds) {
    auto f = a0.tsvd_rounds->find(a0.op_key);
    if (f != a0.tsvd_rounds->end() && f->second > 1) it_cold = TSVD_IT_COLD + ((f->second < 4 ? f->second : 4) - 1) * TSVD_IT_MORE;
  }
  // a block narrower than 2.5 keep converges more slowly: more iterations are still far cheaper than the exact path
  const int it_max = 2 * b >= 5 * keep ? 24 : 72;
  const int max_rounds = 1 + (it_max > it_cold ? (it_max - it_cold + TSVD_IT_MORE - 1) / TSVD_IT_MORE : 0);
  if (keep > 128) return svd_exact(a0, A, US, Vh, work, m, n, keep, nr_bulk, slot_lognorm, slot_trunc);
  Arena a = a0;
  a.mask = nullptr;
  const int64_t q = m < n ? n : m, qp = rup8(q), bb = (int64_t)b * b;
  TsvdBufs w;
  int64_t o = work;
  for (int i = 0; i < 4; ++i) { w.panel[i] = o; o += qp * b; }
  w.X = o; o += b > TSVD_BMAX ? 2 * qp * b + bb : 0;
  w.Gp = o; o += GRAM_SPLIT * bb;
  w.Ri = o; o += bb;      // 1 / diagonal of the last Cholesky factor (b entries) + the inverses of its diagonal blocks
  w.Rs = o; o += bb;      // the last Cholesky factor when the caller does not keep it
  w.R1 = o; o += bb;
  w.R2 = o; o += bb;
  w.Rm = o; o += bb;
  w.Vbs = o; o += 2 * bb; // b x b: all Ritz vectors, rows sorted by singular value
  w.Tk = o; o += bb;      // keep x keep
  w.Pb = o;               // m x n: P = US Vh
  double* stat = a.svd_off;          // [nb] min pivot ratio, then [nb] each: residual, ratio, discarded fraction, [2 nb] norms, partial sums
  double* norms = a.svd_off + 4 * a.nb;
  const cudaGraphConditionalHandle h_loop = new_cond_handle(a), h_exact = new_cond_handle(a);

  // ---- round 1: pseudo-random block, it_cold iterations
  int64_t Qb = w.panel[0], f0 = w.panel[1], f1 = w.panel[2], f2 = w.panel[3];
  PM(7);
  {
    const long long total = (long long)n * b;
    int gx = (int)((total + 255) / 256);
    if (gx > 148 * 4) gx = 148 * 4;
    tsvd_randq_kernel<<<dim3(gx, a.nb), 256, 0, a.stream>>>(a.base, a.chain_stride, Qb, total);
    tsvd_fill_kernel<<<(a.nb + 127) / 128, 128, 0, a.stream>>>(stat, a.nb, 1.0);
    *a.launches += 2;
  }
  auto replace_q = [&](int64_t nq) {
    const int64_t old = Qb;
    Qb = nq;
    if (nq == f0) f0 = old; else if (nq == f1) f1 = old; else f2 = old;
  };
  bool cold_fast = false;
  for (int done = 0; done < it_cold; ++done) {
    gemm(a, f0, A, Qb, m, b, n, OP_N, OP_N);                          // W = A Q          -> f0
    PM(0);
    if (done >= TSVD_SAFE_ITERS) {
      if (!cold_fast) {                                               // pivots of the SAFE start say nothing about the FAST steps
        tsvd_fill_kernel<<<(a.nb + 127) / 128, 128, 0, a.stream>>>(stat, a.nb, 1.0);
        ++*a.launches;
        cold_fast = true;
      }
      gemm(a, f1, A, f0, n, b, m, OP_C, OP_N);                        // Z = A^H W        -> f1
      PM(0);
      cholqr_pass(a, f1, f0, w.Gp, w.Ri, w.Rs, n, b, stat, w.X);           // orth(Z)          -> f0
      if (done + 1 == it_cold) { cholqr_pass(a, f0, f1, w.Gp, w.Ri, w.Rs, n, b, stat, w.X); replace_q(f1); }   // twice on the last one
      else replace_q(f0);
    } else {
      cholqr_pass(a, f0, f1, w.Gp, w.Ri, w.Rs, m, b, stat, w.X);           // Y = orth(W)      -> f1
      gemm(a, f0, A, f1, n, b, m, OP_C, OP_N);                        // Z = A^H Y        -> f0
      PM(0);
      cholqr_pass(a, f0, f1, w.Gp, w.Ri, w.Rs, n, b, stat, w.X);           // orth(Z)          -> f1
      if (done + 1 == it_cold) { cholqr_pass(a, f1, f0, w.Gp, w.Ri, w.Rs, n, b, stat, w.X); replace_q(f0); }   // twice on the last one
      else replace_q(f1);
    }
  }
  if (!cold_fast) {                                                   // all-SAFE schedule: its pivots are not a trust criterion
    tsvd_fill_kernel<<<(a.nb + 127) / 128, 128, 0, a.stream>>>(stat, a.nb, 1.0);
    ++*a.launches;
  }
  rayleigh_ritz_and_check(a, w, A, US, Vh, m, n, keep, b, Qb, f0, f1, cold_fast);
  tsvd_decide_kernel<<<1, 32, 0, a.stream>>>(a.ctl, a.chain_state, stat, a.svd_off + a.nb, a.svd_off + 2 * a.nb, a.svd_off + 3 * a.nb, a.nb, 1,
                                             max_rounds, it_cold, TSVD_IT_MORE, h_loop, h_exact, a.capture ? 1 : 0, a.base, a.chain_stride, w.R1,
                                             b, (int)keep);
  ++*a.launches;

  // ---- further rounds while some chain is RUNNING; only those chains take part
  int rounds = 1;
  if (a.capture) {
    Arena body;
    if (!begin_cond_body(a, h_loop, true, &body)) return -1;
    body.mask = a.chain_state; body.mask_want = CHAIN_RUNNING;
    tsvd_more_round(body, w, A, US, Vh, m, n, keep, b, Qb, f0, f1, f2, max_rounds, it_cold, h_loop, h_exact);
    if (!end_body(body)) return -1;
  } else {
    if (read_ctl(a) != cudaSuccess) return -1;
    t_prof.flush();
    Arena body = a;
    body.mask = a.chain_state; body.mask_want = CHAIN_RUNNING;
    while (a.ctl_host->any_run) {
      if (debug) fprintf(stderr, "[kbp tsvd %lldx%lld keep %lld b %d] round %d: another %d iterations\n", (long long)m, (long long)n, (long long)keep, b, rounds, TSVD_IT_MORE);
      tsvd_more_round(body, w, A, US, Vh, m, n, keep, b, Qb, f0, f1, f2, max_rounds, it_cold, h_loop, h_exact);
      ++rounds;
      if (read_ctl(a) != cudaSuccess) return -1;
      t_prof.flush();
    }
  }
  // ---- accepted chains: scale US, update the slots
  tsvd_finalize_kernel<<<dim3(FIN_CTAS, a.nb), 256, 0, a.stream>>>(a.base, a.chain_stride, a.slots, a.n_slots, US, m * keep, nr_bulk, slot_lognorm, slot_trunc,
                                                                    norms, a.chain_state, CHAIN_ACCEPTED);
  ++*a.launches;
  // ---- chains the iteration could not settle: exact block-Jacobi SVD of the same matrix
  bool used_exact = false;
  if (a.capture) {
    Arena body;
    if (!begin_cond_body(a, h_exact, false, &body)) return -1;
    body.mask = a.chain_state; body.mask_want = CHAIN_EXACT;
    const int r = svd_exact(body, A, US, Vh, work, m, n, keep, nr_bulk, slot_lognorm, slot_trunc);
    if (!end_body(body) || r < 0) return -1;
  } else if (a.ctl_host->any_exact) {
    if (debug) {
      double v[4] = {0, 0, 0, 0};                              // chain 0: pivot ratio, residual, s_keep / s_1, discarded fraction
      for (int q = 0; q < 4; ++q) cudaMemcpy(&v[q], a.svd_off + q * a.nb, sizeof(double), cudaMemcpyDeviceToHost);
      fprintf(stderr, "[kbp tsvd %lldx%lld keep %lld b %d] exact path after %d rounds: residual %.2e  s_keep/s_1 %.2e  discarded fraction %.2e\n", (long long)m,
              (long long)n, (long long)keep, b, rounds, v[1], v[2], v[3]);
    }
    Arena body = a;
    body.mask = a.chain_state; body.mask_want = CHAIN_EXACT;
    if (svd_exact(body, A, US, Vh, work, m, n, keep, nr_bulk, slot_lognorm, slot_trunc) < 0) return -1;
    used_exact = true;
  }
  // what the captured program gives this op: `rounds` iterations up front; 0 = it needed the exact path (keeps its nodes)
  if (!a.capture && a.tsvd_rounds) (*a.tsvd_rounds)[a.op_key] = used_exact ? 0 : rounds;
  return rounds;
}

void qr_householder(const Arena& a, int64_t A, int64_t Q, int64_t R, int64_t work, int64_t m, int64_t n);   // k_qr.cu

bool qr_cholqr2(const Arena& a0, int64_t A, int64_t Q, int64_t R, int64_t work, int64_t m, int64_t n) {
  if (a0.mask != nullptr || n < 8 || n > CREG_BMAX || m < 4 * n) return false;
  const int b = (int)n, nblk = (b + CNB - 1) / CNB;
  const int64_t bb = n * n, need = m * n + GRAM_SPLIT * bb + 2 * bb + n + (int64_t)nblk * CNB * CNB + 8;
  const int64_t k = n;
  if (need > m * n + m * k + k + 8) return false;                  // the op's workspace (kbp_qr_work_elems)
  Arena a = a0;
  const int64_t T1 = work, Gp = T1 + m * n, R1 = Gp + GRAM_SPLIT * bb, R2 = R1 + bb, Dinv = R2 + bb;
  double* stat = a.svd_off;
  tsvd_fill_kernel<<<(a.nb + 127) / 128, 128, 0, a.stream>>>(stat, a.nb, 1.0);
  ++*a.launches;
  cholqr_pass_narrow(a, A, T1, Gp, Dinv, R1, m, b, stat);          // A = Q1 R1
  cholqr_pass_narrow(a, T1, Q, Gp, Dinv, R2, m, b, stat);          // Q1 = Q R2
  gemm(a, R, R2, R1, n, n, n, OP_N, OP_N);                         // R = R2 R1 (upper triangular)
  cholqr2_decide_kernel<<<a.nb, 32, 0, a.stream>>>(a.chain_state, stat, a.base, a.chain_stride, R1, R2, b);
  ++*a.launches;
  // the Householder launches are ALWAYS issued, predicated per chain on the decision above: a chain that passed costs one
  // empty launch.  (An IF node per QR op made concurrently running program graphs serialise each other: six side programs
  // of the N = 6 block went from 730 to 1460 ms per BP iteration.)
  Arena body = a;
  body.mask = a.chain_state;
  body.mask_want = CHAIN_EXACT;
  qr_householder(body, A, Q, R, work, m, n);
  return true;
}

// ------------------------------------------------------------------------------------------------
// QR of a LARGE matrix that is not skinny (m >= n > 96: the 672 x 672 split of the common neighbour in the Mode -> Edge
// reduction at D = 4, src/tensor_networks/tensor_network.py:1194) by block classical Gram-Schmidt with reorthogonalisation:
//   for every block of <= 64 columns:  V = A_j - Q_prev (Q_prev^H A_j), twice;  V = Q_j R_jj by the tall-skinny path (Cholesky-QR
//   twice, Householder per chain if ill conditioned);  R_ij = the two projection coefficients.
// Everything is GEMMs on the DMMA pipe plus the tall QR kernels: ~3 ms against ~150 ms for the one-CTA Householder kernel,
// which was 3/4 of the gate update on the edges whose reduction has this split.  Q is kept TRANSPOSED in the workspace
// (rows = columns of Q, so the blocks found so far are one contiguous matrix for both products).  If any block needed the
// Householder fallback (rank deficient / ill conditioned input: its Q_j is orthonormal but not guaranteed orthogonal to the
// earlier blocks) the chain is redone by the Householder kernels, predicated per chain.
__global__ void qrb_sticky_kernel(double* __restrict__ sticky, const int* __restrict__ state, int nb, int reset) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nb) return;
  if (reset) sticky[c] = 0.0;
  else if (state[c] == CHAIN_EXACT) sticky[c] = 1.0;
}
__global__ void qrb_final_kernel(int* __restrict__ state, const double* __restrict__ sticky, int nb) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < nb) state[c] = sticky[c] != 0.0 ? CHAIN_EXACT : CHAIN_ACCEPTED;
}
// x += y  (n elements)
__global__ void tsvd_add_kernel(cplx* __restrict__ base, long long chain_stride, long long x_, long long y_, long long n) {
  cplx* cb = base + (long long)blockIdx.y * chain_stride;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) cb[x_ + e] = cadd(cb[x_ + e], cb[y_ + e]);
}

void qr(const Arena& a, int64_t A, int64_t Q, int64_t R, int64_t work, int64_t m, int64_t n);

bool qr_blocked(const Arena& a, int64_t A, int64_t Q, int64_t R, int64_t work, int64_t m, int64_t n) {
  if (a.mask != nullptr || m < n || n < 128) return false;
  const int64_t nblocks = (n + 63) / 64;
  const int64_t w = ((n + nblocks - 1) / nblocks + 7) / 8 * 8;         // block width: <= 64, multiple of 8, no tiny last block
  const int64_t Qt = work, V = Qt + n * m, Qj = V + m * w, C1 = Qj + m * w, C2 = C1 + n * w, Rjj = C2 + n * w, wk = Rjj + w * w;
  const int64_t need = (wk - work) + (m * w + m * w + w + 8);
  if (need > m * n + m * n + n + 8) return false;                       // the op's workspace (kbp_qr_work_elems, k = n)
  double* sticky = a.svd_off + 5 * a.nb;
  const int gnb = (a.nb + 127) / 128;
  qrb_sticky_kernel<<<gnb, 128, 0, a.stream>>>(sticky, a.chain_state, a.nb, 1);
  ++*a.launches;
  zero(a, R, n * n);
  for (int64_t c0 = 0; c0 < n; c0 += w) {
    const int64_t wj = c0 + w <= n ? w : n - c0, pj = c0;
    const dim3 gv(grid1d(m * wj), a.nb), gc(grid1d(pj * wj > 0 ? pj * wj : 1), a.nb);
    tsvd_gather_cols_kernel<<<gv, 256, 0, a.stream>>>(a.base, a.chain_stride, V, A, (int)m, (int)n, (int)c0, (int)wj, nullptr, 0);
    ++*a.launches;
    if (pj > 0) {
      gemm(a, C1, Qt, V, pj, wj, m, OP_J, OP_N);                        // Q_prev^H A_j
      gemm(a, Qj, Qt, C1, m, wj, pj, OP_T, OP_N);                       // Q_prev (...)
      tsvd_sub_kernel<<<gv, 256, 0, a.stream>>>(a.base, a.chain_stride, V, Qj, m * wj, nullptr, 0);
      gemm(a, C2, Qt, V, pj, wj, m, OP_J, OP_N);                        // once more (reorthogonalisation)
      gemm(a, Qj, Qt, C2, m, wj, pj, OP_T, OP_N);
      tsvd_sub_kernel<<<gv, 256, 0, a.stream>>>(a.base, a.chain_stride, V, Qj, m * wj, nullptr, 0);
      tsvd_add_kernel<<<gc, 256, 0, a.stream>>>(a.base, a.chain_stride, C1, C2, pj * wj);
      tsvd_scatter_cols_kernel<<<gc, 256, 0, a.stream>>>(a.base, a.chain_stride, R, C1, (int)pj, (int)n, (int)c0, (int)wj, nullptr, 0);
      *a.launches += 4;
    }
    qr(a, V, Qj, Rjj, wk, m, wj);                                       // tall and skinny: Cholesky-QR twice (+ per-chain Householder)
    qrb_sticky_kernel<<<gnb, 128, 0, a.stream>>>(sticky, a.chain_state, a.nb, 0);
    tsvd_scatter_cols_kernel<<<dim3(grid1d(wj * wj), a.nb), 256, 0, a.stream>>>(a.base, a.chain_stride, R + c0 * n, Rjj, (int)wj, (int)n, (int)c0, (int)wj,
                                                                                nullptr, 0);
    *a.launches += 2;
    const int64_t dims[2] = {m, wj}, perm[2] = {1, 0};
    permute(a, Qt + c0 * m, Qj, 0, 2, dims, perm);                      // rows [c0, c0 + wj) of Q^T
  }
  const int64_t dims[2] = {n, m}, perm[2] = {1, 0};
  permute(a, Q, Qt, 0, 2, dims, perm);
  // chains in which some block took the Householder fallback: the whole factorisation again, the stable way
  qrb_final_kernel<<<gnb, 128, 0, a.stream>>>(a.chain_state, sticky, a.nb);
  ++*a.launches;
  Arena body = a;
  body.mask = a.chain_state;
  body.mask_want = CHAIN_EXACT;
  qr_householder(body, A, Q, R, work, m, n);
  return true;
}

void init_tsvd_attributes() {
  cudaFuncSetAttribute(chol_reg_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
  cudaFuncSetAttribute(chol_reg_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
  cudaFuncSetAttribute(chol_reg_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 217 * 1024);
  cudaFuncSetAttribute(chol_blocked_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 217 * 1024);
  cudaFuncSetAttribute(trsm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024);
}

}  // namespace kbp
