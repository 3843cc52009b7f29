// Batched complex128 Householder QR on a thread-block CLUSTER, everything resident in (distributed) shared memory.
//
// The one-CTA kernel in k_qr.cu keeps the matrix in global memory (a 512 x 32 boundary-MPS tensor is 256 KB, more than one
// SM's shared memory) and is bound by what a single SM can pull through L2: ~0.3-0.6 ms per factorisation, every column step
// streaming the trailing matrix twice.  Here the ROWS of A are split over the C CTAs of a cluster (C = 1, 2, 4, 8 so that a
// CTA holds <= 128 rows): CTA r keeps rows [r mloc, (r+1) mloc) of A (later R and the reflectors) and of Q, column-major.
// A Householder step needs two global sums (the column norm; the reflector's inner products with the trailing columns) and
// the back-accumulation of Q one per reflector.  Each is an all-to-all of partial sums between the CTAs: asynchronous DSMEM
// stores that complete a transaction count on the receiver's mbarrier (no cluster barrier), summed in rank order so that all
// CTAs hold bitwise identical totals and build identical reflectors.
//
// Same contract as qr() in k_qr.cu: A(m x n, row-major) = Q(m x r) R(r x n), r = min(m, n), Q^H Q = I also for rank-deficient
// A (boundary MPS tensors are rank deficient on the first swallows of every chain: no Cholesky-type QR), columns that sit
// at 1e-150 do not underflow (sums of squares are carried a second time scaled by 2^400).
#include "kbp_common.cuh"
#include "kbp_ops.cuh"

#include <cooperative_groups.h>
#include <math.h>

namespace cg = cooperative_groups;

namespace kbp {

namespace {

constexpr int QRC_THREADS = 512;
constexpr int QRC_MLOC_MAX = 128;
constexpr size_t QRC_SMEM_MAX = 220 * 1024;
constexpr double QRC_BIG = 2.582249878086908589655919172e120;        // 2^400
constexpr double QRC_TINY2 = 1e-200;                                 // below this a plain sum of squares is not trusted

struct QrcArgs { long long A, Q, R; int m, n; const int* mask; int mask_want; };   // mask: per-chain predicate (kbp_ops.cuh: Arena::mask)

__device__ __forceinline__ uint32_t sm_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t to_rank(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}

struct Xchg {
  double* mine;        // [NV] this CTA's partial sums
  double* tot;         // [NV] totals (identical in every CTA)
  double* xb;          // [2][C][NV] receive buffers
  uint32_t bar0;       // two mbarriers
  int C, rank, NV, tick;
  uint32_t parity;
  bool lost;

  // all threads call; `mine[0..nv)` written by any threads before the call; on return tot[0..nv) is valid for all threads
  __device__ __forceinline__ void run(int nv) {
    const int t = threadIdx.x, nt = blockDim.x;
    __syncthreads();
    if (C == 1) {
      for (int i = t; i < nv; i += nt) tot[i] = mine[i];
      __syncthreads();
      return;
    }
    const int nv2 = (nv + 1) >> 1;                        // 16-byte packets
    if (t == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar0 + 8 * tick), "r"((uint32_t)(C * nv2 * 16)) : "memory");
    for (int idx = t; idx < C * nv2; idx += nt) {
      const int dest = idx % C, k = idx / C;
      const uint32_t dst = to_rank(sm_u32(xb + ((size_t)(tick * C + rank) * NV + 2 * k)), dest);
      const uint32_t rb = to_rank(bar0 + 8 * tick, dest);
      asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f64 [%0], {%1, %2}, [%3];"
                   :: "r"(dst), "d"(mine[2 * k]), "d"(mine[2 * k + 1]), "r"(rb) : "memory");
    }
    uint32_t done = 0;
    for (int spins = 0; !done && spins < (1 << 20); ++spins)
      asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                   : "=r"(done) : "r"(bar0 + 8 * tick), "r"((parity >> tick) & 1u) : "memory");
    if (!done) lost = true;                                // never in a healthy run: bounded spin instead of a hang
    parity ^= 1u << tick;
    for (int i = t; i < nv; i += nt) {
      double s = 0.0;
      for (int r = 0; r < C; ++r) s += xb[(size_t)(tick * C + r) * NV + i];
      tot[i] = s;
    }
    tick ^= 1;
    __syncthreads();
  }
};

// sum over the 16 lanes of a half-warp (every lane gets the total)
__device__ __forceinline__ cplx half_sum(cplx v) {
  const unsigned mask = 0xffffu << (threadIdx.x & 16);     // the two halves of a warp work on different columns (different trip counts)
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) {
    v.x += __shfl_xor_sync(mask, v.x, o);
    v.y += __shfl_xor_sync(mask, v.y, o);
  }
  return v;
}

__global__ void __launch_bounds__(QRC_THREADS) qr_cluster_kernel(cplx* __restrict__ base, long long chain_stride, QrcArgs g) {
  if (g.mask && g.mask[blockIdx.y] != g.mask_want) return;           // the whole cluster of a chain leaves together
  cg::cluster_group cluster = cg::this_cluster();
  const int C = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const int m = g.m, n = g.n, kk = m < n ? m : n;
  const int mloc = (m + C - 1) / C, r0 = rank * mloc;
  const int rows = max(0, min(mloc, m - r0));              // local rows: global index r0 + i
  const int ld = mloc | 1;
  const int NV = (2 * n + 4 + 1) & ~1;
  cplx* W = reinterpret_cast<cplx*>(sm_raw);                                  // [n][ld]   A -> reflectors below / R on and above the diagonal
  cplx* Qm = W + (size_t)n * ld;                                             // [kk][ld]
  double* xb = reinterpret_cast<double*>(Qm + (size_t)kk * ld);               // [2][C][NV]
  double* mine = xb + (size_t)2 * C * NV;                                     // [NV]
  double* tot = mine + NV;                                                    // [NV]
  double* tau = tot + NV;                                                     // [kk]
  double* red = tau + ((kk + 1) & ~1);                                        // [4 * 16 + 2]
  __shared__ __align__(8) unsigned long long bar[2];

  cplx* cb = base + (long long)blockIdx.y * chain_stride;
  const cplx* A = cb + g.A;
  cplx* Q = cb + g.Q;
  cplx* R = cb + g.R;
  const int t = threadIdx.x, nt = blockDim.x, lane = t & 31, w = t >> 5, nw = nt >> 5;
  const int l16 = t & 15, cs = t >> 4, ncs = nt >> 4;      // 16 lanes over the rows of one column, ncs columns at a time

  Xchg X;
  X.mine = mine; X.tot = tot; X.xb = xb; X.bar0 = sm_u32(&bar[0]); X.C = C; X.rank = rank; X.NV = NV; X.tick = 0; X.parity = 0; X.lost = false;
  if (t == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(X.bar0));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(X.bar0 + 8));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (long long e = t; e < (long long)rows * n; e += nt) {
    const int i = (int)(e / n), c = (int)(e - (long long)i * n);
    W[(size_t)c * ld + i] = A[(long long)(r0 + i) * n + c];
  }
  for (int e = t; e < kk * rows; e += nt) {
    const int c = e / rows, i = e - c * rows;
    Qm[(size_t)c * ld + i] = cmake(r0 + i == c ? 1.0 : 0.0, 0.0);
  }
  if (C > 1) cluster.sync(); else __syncthreads();         // barriers initialised and every CTA resident before the first remote store

  // ---------------- forward: R and the reflectors
  for (int j = 0; j < kk; ++j) {
    cplx* x = W + (size_t)j * ld;
    const int jl = j - r0;                                 // local index of the pivot row (owner: 0 <= jl < rows)
    const bool owner = jl >= 0 && jl < rows;
    const int i0 = max(0, jl + 1);                         // local rows below the pivot
    // (1) sum_{i > j} |x_i|^2, plain and with the entries scaled by 2^400
    double s1 = 0.0, s2 = 0.0;
    for (int i = i0 + t; i < rows; i += nt) {
      const cplx v = x[i];
      s1 += cabs2(v);
      const cplx vs = cscale(v, QRC_BIG);
      s2 += cabs2(vs);
    }
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if (lane == 0) { red[2 * w] = s1; red[2 * w + 1] = s2; }
    __syncthreads();
    if (t == 0) {
      double a1 = 0.0, a2 = 0.0;
      for (int k = 0; k < nw; ++k) { a1 += red[2 * k]; a2 += red[2 * k + 1]; }
      mine[0] = a1; mine[1] = a2;
      const cplx al = owner ? x[jl] : cmake(0.0, 0.0);
      mine[2] = al.x; mine[3] = al.y;
    }
    X.run(4);
    // (2) the reflector, identically in every thread of every CTA
    double tj;
    cplx inv_u0, rjj;
    {
      const cplx alpha = cmake(tot[2], tot[3]);
      const bool tiny = !(tot[0] + cabs2(alpha) > QRC_TINY2);
      const double sc = tiny ? QRC_BIG : 1.0;
      const double sg = tiny ? tot[1] : tot[0];
      const cplx as = cscale(alpha, sc);
      const double absa = sqrt(cabs2(as));
      const double nrm = sqrt(fma(absa, absa, sg));
      if (!(nrm > 0.0) || !(nrm < 1e300)) {
        tj = 0.0; inv_u0 = cmake(0.0, 0.0); rjj = alpha;
      } else {
        const cplx ph = absa > 0.0 ? cscale(as, 1.0 / absa) : cmake(1.0, 0.0);
        const double u0 = absa + nrm;                       // |u0| sc : no cancellation
        const double r = sqrt(sg) / u0;                     // <= 1
        tj = 2.0 / (1.0 + r * r);                           // = 2 / (v^H v),  v = x / u0, v_j = 1
        inv_u0 = cscale(cconj(ph), sc / u0);
        rjj = cscale(ph, -nrm / sc);
      }
    }
    if (t == 0) tau[j] = tj;
    for (int i = i0 + t; i < rows; i += nt) x[i] = cmul(x[i], inv_u0);
    if (owner && t == 0 && tj != 0.0) x[jl] = rjj;
    const int ntrail = n - j - 1;
    if (tj == 0.0 || ntrail == 0) { __syncthreads(); continue; }
    __syncthreads();
    // (3) d_c = v^H a_c over the local rows (the pivot row contributes a_jc at its owner)
    for (int c = j + 1 + cs; c < n; c += ncs) {
      const cplx* a = W + (size_t)c * ld;
      cplx d = cmake(0.0, 0.0);
      for (int i = i0 + l16; i < rows; i += 16) d = cadd(d, ccmul(x[i], a[i]));
      d = half_sum(d);
      if (l16 == 0) {
        if (owner) d = cadd(d, a[jl]);
        mine[2 * (c - j - 1)] = d.x;
        mine[2 * (c - j - 1) + 1] = d.y;
      }
    }
    X.run(2 * ntrail);
    // (4) a_c -= tau d_c v
    for (int c = j + 1 + cs; c < n; c += ncs) {
      cplx* a = W + (size_t)c * ld;
      const cplx d = cscale(cmake(tot[2 * (c - j - 1)], tot[2 * (c - j - 1) + 1]), tj);
      for (int i = i0 + l16; i < rows; i += 16) a[i] = csub(a[i], cmul(x[i], d));
      if (owner && l16 == 0) a[jl] = csub(a[jl], d);
    }
    __syncthreads();
  }

  // ---------------- R (kk x n, row-major): each CTA writes the rows it owns
  for (int e = t; e < kk * n; e += nt) {
    const int r = e / n, c = e - r * n, rl = r - r0;
    if (rl >= 0 && rl < rows) R[e] = r <= c ? W[(size_t)c * ld + rl] : cmake(0.0, 0.0);
  }

  // ---------------- backward: Q = H_0 ... H_{kk-1} [I; 0]
  for (int j = kk - 1; j >= 0; --j) {
    const double tj = tau[j];
    if (tj == 0.0) continue;                               // identical everywhere
    const cplx* v = W + (size_t)j * ld;
    const int jl = j - r0;
    const bool owner = jl >= 0 && jl < rows;
    const int i0 = max(0, jl + 1);
    const int nc = kk - j;                                 // columns j .. kk-1 of Q are touched
    for (int c = j + cs; c < kk; c += ncs) {
      const cplx* qc = Qm + (size_t)c * ld;
      cplx d = cmake(0.0, 0.0);
      for (int i = i0 + l16; i < rows; i += 16) d = cadd(d, ccmul(v[i], qc[i]));
      d = half_sum(d);
      if (l16 == 0) {
        if (owner) d = cadd(d, qc[jl]);
        mine[2 * (c - j)] = d.x;
        mine[2 * (c - j) + 1] = d.y;
      }
    }
    X.run(2 * nc);
    for (int c = j + cs; c < kk; c += ncs) {
      cplx* qc = Qm + (size_t)c * ld;
      const cplx d = cscale(cmake(tot[2 * (c - j)], tot[2 * (c - j) + 1]), tj);
      for (int i = i0 + l16; i < rows; i += 16) qc[i] = csub(qc[i], cmul(v[i], d));
      if (owner && l16 == 0) qc[jl] = csub(qc[jl], d);
    }
    __syncthreads();
  }
  for (long long e = t; e < (long long)rows * kk; e += nt) {
    const int i = (int)(e / kk), c = (int)(e - (long long)i * kk);
    Q[(long long)(r0 + i) * kk + c] = X.lost ? cmake(nan(""), 0.0) : Qm[(size_t)c * ld + i];    // a lost exchange must not pass silently
  }
  if (C > 1) cluster.sync();                               // no CTA leaves while others may still address its shared memory
}

size_t qrc_smem(int m, int n, int C) {
  const int kk = m < n ? m : n, mloc = (m + C - 1) / C, ld = mloc | 1, NV = (2 * n + 4 + 1) & ~1;
  return sizeof(double2) * (size_t)(n + kk) * ld + sizeof(double) * ((size_t)2 * C * NV + 2 * NV + ((kk + 1) & ~1) + 4 * 16 + 2) + 64;
}

// smallest cluster (1, 2, 4 or 8 CTAs) whose row slices and shared memory fit, 0 if the shape is not handled here
int qrc_cluster_size(int64_t m, int64_t n) {
  if (m > 8 * QRC_MLOC_MAX || n > 256) return 0;
  int C = 1;
  while (C <= 8 && ((m + C - 1) / C > QRC_MLOC_MAX || qrc_smem((int)m, (int)n, C) > QRC_SMEM_MAX)) C <<= 1;
  return C <= 8 ? C : 0;
}

}  // namespace

// does the cluster kernel take this shape?
bool qr_cluster_fits(int64_t m, int64_t n) { return qrc_cluster_size(m, n) > 0; }

// returns false if the shape is not handled here (caller uses the one-CTA kernel)
bool qr_cluster(const Arena& a, int64_t A, int64_t Q, int64_t R, int64_t m, int64_t n) {
  const int C = qrc_cluster_size(m, n);
  if (C == 0) return false;
  QrcArgs g;
  g.A = A; g.Q = Q; g.R = R; g.m = (int)m; g.n = (int)n; g.mask = a.mask; g.mask_want = a.mask_want;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)C, (unsigned)a.nb);
  cfg.blockDim = dim3(QRC_THREADS);
  cfg.dynamicSmemBytes = qrc_smem((int)m, (int)n, C);
  cfg.stream = a.stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)C;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  if (cudaLaunchKernelEx(&cfg, qr_cluster_kernel, a.base, (long long)a.chain_stride, g) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  ++*a.launches;
  return true;
}

void init_qr_attributes() { cudaFuncSetAttribute(qr_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QRC_SMEM_MAX); }

}  // namespace kbp
