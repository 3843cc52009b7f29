// Simple update (Jiang, Weng and Xiang, PRL 101, 090603 (2008)) of the three-site Kagome unit cell, batched: one CTA per chain
// runs up to max_steps Trotter steps (the six bond updates of the bond table in order) and stops on its own when the largest
// change of a bond's lambda over one step falls below tol.  No host decision inside: the op is one launch whatever the data.
//
// State in the chain's arena slice: Gamma_A, Gamma_B, Gamma_C ([d, D, D, D, D] each, UnitCell leg order) and lambda (6 x D,
// real parts used), updated in place.  One bond update (b = (i, li; j, lj)), everything in shared memory:
//   M_s = Gamma_s with the lambdas of its three other legs absorbed, as [D^3 (other legs), d D (physical, bond leg)]   s = i, j
//   Householder QR of both: M_s = Q_s R_s, the reflectors kept in place of M_s
//   theta[(a, p'), (b, q')] = sum g[p', p, q', q] R_i[a, (p, k)] lambda_b[k] R_j[b, (q, k)]        (d^2 D x d^2 D)
//   one-sided Jacobi on the rows of [theta | I] (the helpers of the small SVD, kbp_jacobi.cuh): rows converge to
//   [s_k Vh_k | U_k^H];  keep the D largest
//   lambda_b = s[:D] / |s[:D]|,  Gamma_i = Q_i U,  Gamma_j = Q_j conj(V)  (reflectors applied to [Y; 0]),  other legs' lambdas
//   divided back out (zero inverse below SU_LAMBDA_CUTOFF * max), both scaled to unit Frobenius norm
// At the end every bond's two-site RDM in the SU environment (lambda on all outer legs, ket and bra) is written, [i, i*, j, j*],
// unit trace, from the Gram matrices M_s^H M_s.  The numpy statement of the same algorithm is oracle/su_np.py.
#include "kbp_common.cuh"
#include "kbp_jacobi.cuh"
#include "kbp_ops.cuh"

#include <math.h>
#include <string.h>

namespace kbp {

constexpr double SU_LAMBDA_CUTOFF = 1e-12;   // oracle/su_np.py: LAMBDA_CUTOFF
constexpr int SU_MAX_SWEEPS = 60;
constexpr int SU_THREADS = 384;              // 12 warps: one per row pair of the largest theta (24 rows at D = 6)

struct SuLayout {
  int m, n, p, q;                  // M: m x n;  theta rows p, [theta | I] row length q
  size_t off_M[2], off_Z[2], off_X, off_beta, off_alpha, off_s2, off_idx, off_rec, off_lam, off_gate, total;
};

__host__ __device__ inline SuLayout su_layout(int d, int D) {
  SuLayout L;
  L.m = D * D * D; L.n = d * D; L.p = d * L.n; L.q = 2 * L.p;
  size_t o = 0;
  auto take = [&](size_t bytes) { const size_t r = o; o += (bytes + 15) & ~(size_t)15; return r; };
  const size_t mn = sizeof(cplx) * (size_t)L.m * L.n;
  L.off_M[0] = take(mn); L.off_M[1] = take(mn);
  L.off_Z[0] = take(mn); L.off_Z[1] = take(mn);
  L.off_X = take(sizeof(cplx) * (size_t)L.p * L.q);
  L.off_beta = take(sizeof(double) * 2 * L.n);
  L.off_alpha = take(sizeof(cplx) * 2 * L.n);
  L.off_s2 = take(sizeof(double) * L.p);
  L.off_idx = take(sizeof(int) * L.p);
  L.off_rec = take(sizeof(PairSums) * (L.p / 2));
  L.off_lam = take(sizeof(double) * 7 * D);       // 6 bonds + the old lambda of the bond in flight
  L.off_gate = take(sizeof(cplx) * d * d * d * d);
  L.total = o;
  return L;
}

struct SuArgs {
  long long G[3], lam, gate, rdm;   // arena offsets
  int d, D, max_steps;
  double tol;
  int slot_steps, slot_delta, slot_nonfinite;
  int bi[6], li[6], bj[6], lj[6];
};

// element e of Gamma [p, l0, l1, l2, l3] -> (row = other legs of `leg` in leg order, col = p D + l_leg) and the four leg indices
__device__ __forceinline__ void su_split(int e, int D, int leg, int& row, int& col, int (&l)[4]) {
#pragma unroll
  for (int k = 3; k >= 0; --k) { l[k] = e % D; e /= D; }
  row = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (k != leg) row = row * D + l[k];
  col = e * D + l[leg];
}

__device__ __forceinline__ double su_inv(double x, double mx) { return x > SU_LAMBDA_CUTOFF * mx ? 1.0 / x : 0.0; }

// M_s (m x n) = Gamma_s with the lambdas of its other legs absorbed, for both ends of bond b
__device__ void su_load_pair(const cplx* const* G, const double* lam, const int (&legb)[3][4], int D, int elems, const int (&site)[2],
                             const int (&leg)[2], cplx* const (&M)[2], int n) {
  for (int t = threadIdx.x; t < 2 * elems; t += blockDim.x) {
    const int s = t >= elems, e = t - s * elems;
    int row, col, l[4];
    su_split(e, D, leg[s], row, col, l);
    double w = 1.0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (k != leg[s]) w *= lam[legb[site[s]][k] * D + l[k]];
    M[s][row * n + col] = cscale(G[site[s]][e], w);
  }
  __syncthreads();
}

__global__ void __launch_bounds__(SU_THREADS) su_kernel(cplx* __restrict__ base, long long chain_stride, double* __restrict__ slots, int n_slots,
                                                        SuArgs g) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  __shared__ double red[34];
  __shared__ int legb_s[3][4];
  __shared__ double delta_s;
  const int d = g.d, D = g.D;
  const SuLayout L = su_layout(d, D);
  const int m = L.m, n = L.n, p = L.p, q = L.q, elems = d * D * D * D * D;
  cplx* const M[2] = {reinterpret_cast<cplx*>(sm_raw + L.off_M[0]), reinterpret_cast<cplx*>(sm_raw + L.off_M[1])};
  cplx* const Z[2] = {reinterpret_cast<cplx*>(sm_raw + L.off_Z[0]), reinterpret_cast<cplx*>(sm_raw + L.off_Z[1])};
  cplx* X = reinterpret_cast<cplx*>(sm_raw + L.off_X);
  double* beta = reinterpret_cast<double*>(sm_raw + L.off_beta);      // [2][n]
  cplx* alpha = reinterpret_cast<cplx*>(sm_raw + L.off_alpha);        // [2][n]  diagonal of R
  double* s2 = reinterpret_cast<double*>(sm_raw + L.off_s2);
  int* idx = reinterpret_cast<int*>(sm_raw + L.off_idx);
  PairSums* rec = reinterpret_cast<PairSums*>(sm_raw + L.off_rec);
  double* lam = reinterpret_cast<double*>(sm_raw + L.off_lam);        // [6][D], then the old lambda of the bond in flight
  double* lam_old = lam + 6 * D;
  cplx* gate = reinterpret_cast<cplx*>(sm_raw + L.off_gate);

  cplx* cb = base + (long long)blockIdx.x * chain_stride;
  cplx* const G[3] = {cb + g.G[0], cb + g.G[1], cb + g.G[2]};
  cplx* lam_g = cb + g.lam;
  const int t = threadIdx.x, nt = blockDim.x, lane = t & 31, w = t >> 5, nw = nt >> 5;

  for (int k = t; k < 6 * D; k += nt) lam[k] = lam_g[k].x;
  for (int k = t; k < d * d * d * d; k += nt) gate[k] = cb[g.gate + k];
  if (t < 6) { legb_s[g.bi[t]][g.li[t]] = t; legb_s[g.bj[t]][g.lj[t]] = t; }
  __syncthreads();
  int legb[3][4];
#pragma unroll
  for (int s = 0; s < 3; ++s)
#pragma unroll
    for (int k = 0; k < 4; ++k) legb[s][k] = legb_s[s][k];

  auto Rval = [&](int s, int r, int c) -> cplx { return c > r ? M[s][r * n + c] : (c == r ? alpha[s * n + r] : cmake(0.0, 0.0)); };

  int steps = 0;
  double delta = 0.0;
  bool finite = true;
  while (steps < g.max_steps) {
    double step_delta = 0.0;
    for (int b = 0; b < 6 && finite; ++b) {
      const int site[2] = {g.bi[b], g.bj[b]}, leg[2] = {g.li[b], g.lj[b]};
      su_load_pair(G, lam, legb, D, elems, site, leg, M, n);

      // ---- Householder QR of M_0 and M_1 side by side.  P = I - beta u u^H with u = x - alpha e1, alpha = -e^{i arg x0} |x|
      for (int k = 0; k < n; ++k) {
        if (w < 2) {
          cplx* Ms = M[w];
          double acc = 0.0;
          for (int r = k + lane; r < m; r += 32) acc += cabs2(Ms[r * n + k]);
          const double nx = sqrt(warp_sum(acc));
          if (lane == 0) {
            const cplx x0 = Ms[k * n + k];
            const double a0 = sqrt(cabs2(x0));
            const cplx e = a0 > 0.0 ? cscale(x0, 1.0 / a0) : cmake(1.0, 0.0);
            alpha[w * n + k] = cscale(e, -nx);
            Ms[k * n + k] = cscale(e, a0 + nx);                     // u0 = x0 - alpha
            beta[w * n + k] = nx > 0.0 ? 1.0 / (nx * (nx + a0)) : 0.0;   // 2 / u^H u
          }
        }
        __syncthreads();
        const int ncol = n - k - 1;
        for (int task = w; task < 2 * ncol; task += nw) {
          const int s = task >= ncol, c = k + 1 + task - s * ncol;
          cplx* Ms = M[s];
          cplx acc = cmake(0.0, 0.0);
          for (int r = k + lane; r < m; r += 32) acc = cadd(acc, ccmul(Ms[r * n + k], Ms[r * n + c]));
          acc = cscale(warp_sum(acc), beta[s * n + k]);
          for (int r = k + lane; r < m; r += 32) Ms[r * n + c] = csub(Ms[r * n + c], cmul(Ms[r * n + k], acc));
        }
        __syncthreads();
      }

      // ---- [theta | I]
      for (int e = t; e < p * p; e += nt) {
        const int row = e / p, col = e - row * p;
        const int a = row / d, P = row - a * d, bb = col / d, Q = col - bb * d;
        cplx acc = cmake(0.0, 0.0);
        for (int pp = 0; pp < d; ++pp)
          for (int qq = 0; qq < d; ++qq) {
            const cplx gv = gate[((P * d + pp) * d + Q) * d + qq];
            if (gv.x == 0.0 && gv.y == 0.0) continue;
            cplx th = cmake(0.0, 0.0);
            for (int k = 0; k < D; ++k)
              th = cfma(cscale(Rval(0, a, pp * D + k), lam[b * D + k]), Rval(1, bb, qq * D + k), th);
            acc = cfma(gv, th, acc);
          }
        X[row * q + col] = acc;
        X[row * q + p + col] = cmake(row == col ? 1.0 : 0.0, 0.0);
      }
      for (int k = t; k < D; k += nt) lam_old[k] = lam[b * D + k];
      double fro = 0.0;
      for (int e = t; e < p * p; e += nt) fro += cabs2(X[(e / p) * q + e % p]);
      const double floor2 = 1e-34 * block_sum(fro, red);        // (barrier: X published)

      // ---- one-sided Jacobi on the rows of [theta | I], one warp per row pair
      {
        const int npairs = p / 2;
        const unsigned gmask = 0xffffffffu;
        bool converged = false;
        for (int sweep = 0; sweep < SU_MAX_SWEEPS && !converged; ++sweep) {
          bool big = false;
          PairWalk walk;
          walk.start(p, w);
          for (int step = 0; step < p - 1; ++step) {
            int i, j;
            walk.get(step, i, j);
            if (w < npairs) {
              if (q <= 32) jacobi_pair_cached<1, 32>(X + i * q, X + j * q, q, p, lane, gmask, floor2, big, rec + w);
              else jacobi_pair_cached<2, 32>(X + i * q, X + j * q, q, p, lane, gmask, floor2, big, rec + w);
            }
            walk.next();
            __syncthreads();
          }
          converged = !__syncthreads_or(big ? 1 : 0);
        }
      }

      // ---- singular values, rank sort (descending, stable), new lambda_b
      for (int i = w; i < p; i += nw) {
        double acc = 0.0;
        for (int c = lane; c < p; c += 32) acc += cabs2(X[i * q + c]);
        acc = warp_sum(acc);
        if (lane == 0) s2[i] = acc;
      }
      __syncthreads();
      for (int i = t; i < p; i += nt) {
        const double si = s2[i];
        int rank = 0;
        for (int j = 0; j < p; ++j) rank += (s2[j] > si) || (s2[j] == si && j < i);
        idx[rank] = i;
      }
      __syncthreads();
      if (t == 0) {
        double kept = 0.0;
        for (int k = 0; k < D; ++k) kept += s2[idx[k]];
        const double rn = kept > 0.0 ? 1.0 / sqrt(kept) : 0.0;
        double dl = 0.0;
        for (int k = 0; k < D; ++k) {
          const double v = sqrt(s2[idx[k]]) * rn;
          dl += (v - lam_old[k]) * (v - lam_old[k]);
          lam[b * D + k] = v;
          lam_g[b * D + k] = cmake(v, 0.0);
        }
        delta_s = sqrt(dl);
      }

      // ---- Y_i[a, (p', k)] = U[(a, p'), k],  Y_j[b, (q', k)] = conj(V)[(b, q'), k];  Z_s = [Y_s; 0]
      for (int e = t; e < 2 * m * n; e += nt) {
        const int s = e >= m * n, r = (e - s * m * n) / n, c = (e - s * m * n) - r * n;
        cplx v = cmake(0.0, 0.0);
        if (r < n) {
          const int P = c / D, k = c - P * D, row = idx[k];
          if (s == 0) v = cconj(X[row * q + p + r * d + P]);
          else v = s2[row] > floor2 ? cscale(X[row * q + r * d + P], rsqrt(s2[row])) : cmake(0.0, 0.0);
        }
        Z[s][r * n + c] = v;
      }
      __syncthreads();
      // ---- Z_s = Q_s Y_s = P_0 ... P_{n-1} [Y_s; 0]
      for (int k = n - 1; k >= 0; --k) {
        for (int task = w; task < 2 * n; task += nw) {
          const int s = task >= n, c = task - s * n;
          const cplx* u = M[s];
          cplx* Zs = Z[s];
          cplx acc = cmake(0.0, 0.0);
          for (int r = k + lane; r < m; r += 32) acc = cadd(acc, ccmul(u[r * n + k], Zs[r * n + c]));
          acc = cscale(warp_sum(acc), beta[s * n + k]);
          for (int r = k + lane; r < m; r += 32) Zs[r * n + c] = csub(Zs[r * n + c], cmul(u[r * n + k], acc));
        }
        __syncthreads();
      }

      // ---- Gamma_s = Z_s with the other legs' lambdas divided out, unit norm
      double mx[2][4];
#pragma unroll
      for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          double v = 0.0;
          if (k != leg[s]) for (int x = 0; x < D; ++x) v = fmax(v, lam[legb[site[s]][k] * D + x]);
          mx[s][k] = v;
        }
      double nrm[2];
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        double acc = 0.0;
        for (int e = t; e < elems; e += nt) {
          int row, col, l[4];
          su_split(e, D, leg[s], row, col, l);
          double wt = 1.0;
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (k != leg[s]) wt *= su_inv(lam[legb[site[s]][k] * D + l[k]], mx[s][k]);
          acc += cabs2(Z[s][row * n + col]) * wt * wt;
        }
        nrm[s] = block_sum(acc, red);
      }
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const double sc = nrm[s] > 0.0 ? 1.0 / sqrt(nrm[s]) : 0.0;
        for (int e = t; e < elems; e += nt) {
          int row, col, l[4];
          su_split(e, D, leg[s], row, col, l);
          double wt = sc;
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (k != leg[s]) wt *= su_inv(lam[legb[site[s]][k] * D + l[k]], mx[s][k]);
          G[site[s]][e] = cscale(Z[s][row * n + col], wt);
        }
      }
      __syncthreads();                                   // Gamma (global) and lambda visible to the next bond
      const double db = delta_s;
      finite = db == db && db <= 1e300;
      step_delta = fmax(step_delta, db);
      __syncthreads();
    }
    ++steps;
    delta = finite ? step_delta : __longlong_as_double(0x7ff8000000000000LL);
    if (!finite || delta < g.tol) break;
  }

  // ---- SU-environment RDM of every bond from the Gram matrices of M_i, M_j
  cplx* Gm = X;                                          // [2][n][n]
  for (int b = 0; b < 6; ++b) {
    const int site[2] = {g.bi[b], g.bj[b]}, leg[2] = {g.li[b], g.lj[b]};
    su_load_pair(G, lam, legb, D, elems, site, leg, M, n);
    for (int e = t; e < 2 * n * n; e += nt) {
      const int s = e >= n * n, r = (e - s * n * n) / n, c = (e - s * n * n) - r * n;
      cplx acc = cmake(0.0, 0.0);
      for (int o = 0; o < m; ++o) acc = cadd(acc, cmulc(M[s][o * n + r], M[s][o * n + c]));
      Gm[e] = acc;                                       // Gm_s[(p, k), (p*, k')] = sum_o M_s[o, (p, k)] conj(M_s[o, (p*, k')])
    }
    __syncthreads();
    cplx* rho = Gm + 2 * n * n;                          // d^4
    for (int e = t; e < d * d * d * d; e += nt) {
      const int P = e / (d * d * d), Ps = (e / (d * d)) % d, Q = (e / d) % d, Qs = e % d;
      cplx acc = cmake(0.0, 0.0);
      for (int k = 0; k < D; ++k)
        for (int k2 = 0; k2 < D; ++k2)
          acc = cfma(cscale(Gm[(P * D + k) * n + Ps * D + k2], lam[b * D + k] * lam[b * D + k2]), Gm[n * n + (Q * D + k) * n + Qs * D + k2], acc);
      rho[e] = acc;
    }
    __syncthreads();
    cplx tr = cmake(0.0, 0.0);
    for (int P = 0; P < d; ++P)
      for (int Q = 0; Q < d; ++Q) tr = cadd(tr, rho[((P * d + P) * d + Q) * d + Q]);
    const double den = cabs2(tr);
    const cplx inv = den > 0.0 ? cmake(tr.x / den, -tr.y / den) : cmake(0.0, 0.0);
    for (int e = t; e < d * d * d * d; e += nt) cb[g.rdm + b * d * d * d * d + e] = cmul(rho[e], inv);
    __syncthreads();
  }

  // ---- slots: steps done, last delta, non-finite entries of the state and the RDMs
  double bad = 0.0;
  for (int e = t; e < 3 * elems; e += nt) {
    const cplx v = G[e / elems][e % elems];
    bad += !(isfinite(v.x) && isfinite(v.y));
  }
  for (int e = t; e < 6 * D + 6 * d * d * d * d; e += nt) {
    const cplx v = e < 6 * D ? lam_g[e] : cb[g.rdm + e - 6 * D];
    bad += !(isfinite(v.x) && isfinite(v.y));
  }
  bad = block_sum(bad, red);
  if (t == 0) {
    double* sl = slots + (long long)blockIdx.x * n_slots;
    if (g.slot_steps >= 0) sl[g.slot_steps] = steps;
    if (g.slot_delta >= 0) sl[g.slot_delta] = delta;
    if (g.slot_nonfinite >= 0) sl[g.slot_nonfinite] = bad;
  }
}

size_t su_smem_bytes(int d, int D) { return su_layout(d, D).total; }

bool su_supported(int d, int D) { return d == 2 && D >= 2 && D <= 6; }

void simple_update(const Arena& a, const int64_t* w) {
  SuArgs g;
  g.G[0] = w[0]; g.G[1] = w[1]; g.G[2] = w[2]; g.lam = w[3]; g.gate = w[4]; g.rdm = w[5];
  g.d = (int)w[6]; g.D = (int)w[7]; g.max_steps = (int)w[8];
  memcpy(&g.tol, &w[9], sizeof(double));
  g.slot_steps = (int)w[10]; g.slot_delta = (int)w[11]; g.slot_nonfinite = (int)w[12];
  for (int b = 0; b < 6; ++b) { g.bi[b] = (int)w[13 + 4 * b]; g.li[b] = (int)w[14 + 4 * b]; g.bj[b] = (int)w[15 + 4 * b]; g.lj[b] = (int)w[16 + 4 * b]; }
  su_kernel<<<a.nb, SU_THREADS, su_smem_bytes(g.d, g.D), a.stream>>>(a.base, a.chain_stride, a.slots, a.n_slots, g);
  ++*a.launches;
}

void init_su_attributes() {
  cudaFuncSetAttribute(su_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)su_smem_bytes(2, 6));
}

}  // namespace kbp
