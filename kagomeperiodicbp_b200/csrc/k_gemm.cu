// Batched complex128 GEMM on the FP64 tensor pipe (DMMA m16n8k8):  C = opA(A) * opB(B), row-major.
//
// The boundary-MPS chain is a long sequence of SMALL dependent products (m, n of a few hundred at most,
// k up to a few thousand), so what bounds a product is latency, not the tensor pipe: one CTA computes a
// BM x BN tile with 8 warps and streams its k-slabs through a 3- or 4-stage cp.async ring in shared memory
// (16-byte copies of whole complex128 elements, zero-filled past the edges), one barrier per slab.
// Tiles are 64x64 (warps 4 x 2, four 16x8 accumulators each) when that already fills the machine, else
// 32x32 (warps 2 x 4), else 16x16 (2 warps); products with a long k and a tiny output (Gram matrices Y^H Y) can additionally be
// split along k into `ksplit` partial results written side by side (summed by the consumer: deterministic,
// no atomics).  Operands stay in the layout they have in HBM -- "k-contiguous" [row][k] or
// "m-contiguous" [k][row] depending on op -- so every copy is coalesced and transposition / conjugation
// happen in the fragment loads: one LDS.128 brings (re, im) of an element, conflict-free for both layouts
// (row strides of 20 resp. BM+2 elements).  The complex product is THREE real DMMAs per (tile, k8) (3M form, see the kernel).
#include "kbp_common.cuh"
#include "kbp_ops.cuh"

#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

namespace kbp {

constexpr int BK = 16;
constexpr int LDK = BK + 4;       // row stride (elements) of a k-contiguous tile

struct GemmArgs {
  long long C, A, B;
  int m, n, k, opA, opB;
  int ksplit;                     // partial results: C + s * m * n, s < ksplit
  int rows_on_x;                  // grid.x (2^31 limit) carries the row tiles instead of the column tiles
  int fused;                      // ksplit > 1 only: partials go to the scratch area and the LAST CTA of every tile adds them up
  double2* scratch;               // [nb][scratch_stride]
  long long scratch_stride;
  int* counters;                  // [nb][GEMM_MAX_TILES], zero between launches
  const int* mask;                // per-chain predicate (kbp_ops.cuh: Arena::mask)
  int mask_want;
  int ktime_slot;                 // developer probe (KBP_KTIME=1): slot of this launch in the device time table, -1 = off
};

// developer probe: first CTA start / last CTA end of every GEMM launch by %globaltimer (KBP_KTIME=1)
constexpr int GEMM_KT_SLOTS = 1 << 16;
__device__ unsigned long long g_gemm_t0[GEMM_KT_SLOTS], g_gemm_t1[GEMM_KT_SLOTS];
__device__ __forceinline__ unsigned long long gemm_globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

constexpr int GEMM_MAX_TILES = 4096;
constexpr int GEMM_WARPS_TARGET = 900;    // automatic split-K: warps a small product is split up to

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool valid) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

template <int BM, int BN, int STAGES, int NWARPS, bool A_KC, bool B_KC>
__global__ void __launch_bounds__(32 * NWARPS) zgemm_dmma_kernel(cplx* __restrict__ base, long long chain_stride, GemmArgs g) {
  constexpr int NTHR = 32 * NWARPS;
  constexpr int WMS = BM / 16, WNS = NWARPS / WMS;    // warp grid
  constexpr int NT = BN / WNS / 8;               // 16x8 accumulator tiles per warp
  constexpr int TA = (BM * LDK > BK * (BM + 2)) ? BM * LDK : BK * (BM + 2);   // elements per A tile (either layout)
  constexpr int TB = (BN * LDK > BK * (BN + 2)) ? BN * LDK : BK * (BN + 2);
  constexpr int LDM = BM + 2, LDN = BN + 2;
  extern __shared__ __align__(16) unsigned char gemm_smem[];
  cplx* As = reinterpret_cast<cplx*>(gemm_smem);                 // [STAGES][TA]
  cplx* Bs = As + STAGES * TA;                                   // [STAGES][TB]

  const int chain = blockIdx.z / g.ksplit, split = blockIdx.z - chain * g.ksplit;
  if (g.mask && g.mask[chain] != g.mask_want) return;
  if (g.ktime_slot >= 0 && threadIdx.x == 0) atomicMin(&g_gemm_t0[g.ktime_slot], gemm_globaltimer());
  cplx* Cb = base + (long long)chain * chain_stride + g.C + (long long)split * g.m * g.n;
  const cplx* Ab = base + (long long)chain * chain_stride + g.A;
  const cplx* Bb = base + (long long)chain * chain_stride + g.B;
  const int row0 = (g.rows_on_x ? blockIdx.x : blockIdx.y) * BM, col0 = (g.rows_on_x ? blockIdx.y : blockIdx.x) * BN;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const int wm = w % WMS, wn = w / WMS;
  const int gq = lane >> 2, q = lane & 3;
  constexpr bool a_kc = A_KC;                           // A stored [m][k]  (opA == N or J)
  constexpr bool b_kc = B_KC;                           // B stored [n][k]  (opB == T or C)
  // conjugation = sign flip of the imaginary part, as an integer XOR on the high word (a multiplication by +-1 would be one more
  // instruction on the FP64 pipe per loaded element, the pipe the DMMAs need)
  const int sa = (g.opA == OP_C || g.opA == OP_J) ? (int)0x80000000 : 0;
  const int sb = (g.opB == OP_C || g.opB == OP_J) ? (int)0x80000000 : 0;
  auto flip = [](double y, int bits) { return __hiloint2double(__double2hiint(y) ^ bits, __double2loint(y)); };

  const int slabs_total = (g.k + BK - 1) / BK;
  const int per = (slabs_total + g.ksplit - 1) / g.ksplit;
  const int s_begin = split * per;
  int s_end = s_begin + per;
  if (s_end > slabs_total) s_end = slabs_total;
  const int nslab = s_end > s_begin ? s_end - s_begin : 0;

  // global -> shared copies: every thread owns RA + RB fixed (row, k) positions of a slab.  Source pointers, shared-memory
  // offsets and row validity are computed ONCE; a slab advances the pointers by a constant (the address arithmetic and
  // bounds tests per copy were most of the instructions of a small product, whose warps are bound by dependent issue)
  constexpr int RA = BM * BK / NTHR, RB = BN * BK / NTHR;
  const cplx* pa[RA];
  const cplx* pb[RB];
  int oa[RA], ob[RB], ka[RA], kb[RB];                  // shared offset; k - (k index inside the slab): copy valid iff k0 < ka
  const long long stepA = a_kc ? BK : (long long)BK * g.m, stepB = b_kc ? BK : (long long)BK * g.n;
#pragma unroll
  for (int r = 0; r < RA; ++r) {
    const int c = t + NTHR * r;
    const int mm = a_kc ? c / BK : c % BM, kk = a_kc ? c % BK : c / BM;
    const bool rowok = row0 + mm < g.m;
    oa[r] = a_kc ? mm * LDK + kk : kk * LDM + mm;
    ka[r] = rowok ? g.k - kk : 0;
    pa[r] = Ab + (a_kc ? (long long)(rowok ? row0 + mm : 0) * g.k + (long long)s_begin * BK + kk
                       : ((long long)s_begin * BK + kk) * g.m + (rowok ? row0 + mm : 0));
  }
#pragma unroll
  for (int r = 0; r < RB; ++r) {
    const int c = t + NTHR * r;
    const int nn = b_kc ? c / BK : c % BN, kk = b_kc ? c % BK : c / BN;
    const bool colok = col0 + nn < g.n;
    ob[r] = b_kc ? nn * LDK + kk : kk * LDN + nn;
    kb[r] = colok ? g.k - kk : 0;
    pb[r] = Bb + (b_kc ? (long long)(colok ? col0 + nn : 0) * g.k + (long long)s_begin * BK + kk
                       : ((long long)s_begin * BK + kk) * g.n + (colok ? col0 + nn : 0));
  }
  auto issue = [&](int slab, int stage) {
    const int k0 = (s_begin + slab) * BK;
    cplx* at = As + stage * TA;
    cplx* bt = Bs + stage * TB;
#pragma unroll
    for (int r = 0; r < RA; ++r) {
      const bool ok = k0 < ka[r];
      cp_async16(at + oa[r], ok ? pa[r] + slab * stepA : Ab, ok);
    }
#pragma unroll
    for (int r = 0; r < RB; ++r) {
      const bool ok = k0 < kb[r];
      cp_async16(bt + ob[r], ok ? pb[r] + slab * stepB : Bb, ok);
    }
  };

  // The complex product takes THREE real DMMAs per (tile, k8) instead of four (the "3M" form):
  //     P1 += Ar Br ;  P2 += Ai Bi ;  P3 += (Ar + Ai)(Br + Bi)        ->   Cr = P1 - P2 ,  Ci = P3 - P1 - P2
  // -- a quarter less work on the FP64 pipe, which DMMA shares with every DFMA of the one-SM kernels running beside the
  // products of other chains; the two fragment sums cost one DADD per loaded element.  Normwise as accurate as the four-product
  // form (|dC| <~ k eps |A| |B|).  FP64 DMMA also has a long dependent-issue latency: the three products are independent
  // chains, and the small-tile configurations (NT <= 2) keep a second set for the odd k8 steps, added up in the epilogue.
  constexpr int NACC = (NT <= 2) ? 2 : 1;
  double p1[NACC][NT][4], p2[NACC][NT][4], p3[NACC][NT][4];
#pragma unroll
  for (int q4 = 0; q4 < NACC; ++q4)
#pragma unroll
    for (int i = 0; i < NT; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) p1[q4][i][j] = p2[q4][i][j] = p3[q4][i][j] = 0.0;

#pragma unroll
  for (int s = 0; s < STAGES - 1; ++s) {
    if (s < nslab) issue(s, s);
    cp_async_commit();
  }
  for (int slab = 0; slab < nslab; ++slab) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();                                   // slab's data visible; everyone finished slab-1's stage
    if (slab + STAGES - 1 < nslab) issue(slab + STAGES - 1, (slab + STAGES - 1) % STAGES);
    cp_async_commit();
    const cplx* at = As + (slab % STAGES) * TA;
    const cplx* bt = Bs + (slab % STAGES) * TB;
#pragma unroll
    for (int ks = 0; ks < BK / 8; ++ks) {
      double ar[4], aim[4], as[4];
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int mm = wm * 16 + gq + 8 * (v & 1), kk = ks * 8 + q + 4 * (v >> 1);
        const cplx x = a_kc ? at[mm * LDK + kk] : at[kk * LDM + mm];
        ar[v] = x.x;
        aim[v] = flip(x.y, sa);
        as[v] = ar[v] + aim[v];
      }
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        double br[2], bi[2], bs[2];
#pragma unroll
        for (int v = 0; v < 2; ++v) {
          const int kk = ks * 8 + q + 4 * v, nn = wn * (NT * 8) + nt * 8 + gq;
          const cplx x = b_kc ? bt[nn * LDK + kk] : bt[kk * LDN + nn];
          br[v] = x.x;
          bi[v] = flip(x.y, sb);
          bs[v] = br[v] + bi[v];
        }
        const int a0 = NACC == 2 ? (ks & 1) : 0;
        dmma16x8x8(p1[a0][nt], ar, br);
        dmma16x8x8(p2[a0][nt], aim, bi);
        dmma16x8x8(p3[a0][nt], as, bs);
      }
    }
  }
  cp_async_wait<0>();
  if (g.ktime_slot >= 0 && threadIdx.x == 0) atomicMax(&g_gemm_t1[g.ktime_slot], gemm_globaltimer());   // (epilogue not included)
  if (g.fused) {
    // split-K without a second launch: every CTA parks its partial tile, the last one to arrive at the tile's counter adds
    // the ksplit partials in fixed order (bitwise deterministic) and writes C
    __shared__ int sh_last;
    cplx* part = g.scratch + (long long)chain * g.scratch_stride;
    const long long mn = (long long)g.m * g.n;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int r = row0 + wm * 16 + gq + 8 * (v >> 1);
        const int c = col0 + wn * (NT * 8) + nt * 8 + 2 * q + (v & 1);
        double s1 = p1[0][nt][v], s2 = p2[0][nt][v], s3 = p3[0][nt][v];
#pragma unroll
        for (int q4 = 1; q4 < NACC; ++q4) { s1 += p1[q4][nt][v]; s2 += p2[q4][nt][v]; s3 += p3[q4][nt][v]; }
        const double sr = s1 - s2, si = (s3 - s1) - s2;
        if (r < g.m && c < g.n) part[split * mn + (long long)r * g.n + c] = cmake(sr, si);
      }
    __threadfence();
    __syncthreads();
    const int tile = blockIdx.y * gridDim.x + blockIdx.x;
    if (t == 0) sh_last = atomicAdd(g.counters + chain * GEMM_MAX_TILES + tile, 1) == g.ksplit - 1;
    __syncthreads();
    if (!sh_last) return;
    __threadfence();
    Cb = base + (long long)chain * chain_stride + g.C;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        const int r = row0 + wm * 16 + gq + 8 * (v >> 1);
        const int c = col0 + wn * (NT * 8) + nt * 8 + 2 * q + (v & 1);
        if (r < g.m && c < g.n) {
          double sr = 0.0, si = 0.0;
          for (int sp = 0; sp < g.ksplit; ++sp) {
            const cplx x = __ldcg(part + sp * mn + (long long)r * g.n + c);
            sr += x.x; si += x.y;
          }
          Cb[(long long)r * g.n + c] = cmake(sr, si);
        }
      }
    if (t == 0) g.counters[chain * GEMM_MAX_TILES + tile] = 0;
    return;
  }
#pragma unroll
  for (int nt = 0; nt < NT; ++nt)
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int r = row0 + wm * 16 + gq + 8 * (v >> 1);
      const int c = col0 + wn * (NT * 8) + nt * 8 + 2 * q + (v & 1);
      double s1 = p1[0][nt][v], s2 = p2[0][nt][v], s3 = p3[0][nt][v];
#pragma unroll
      for (int q4 = 1; q4 < NACC; ++q4) { s1 += p1[q4][nt][v]; s2 += p2[q4][nt][v]; s3 += p3[q4][nt][v]; }
      const double sr = s1 - s2, si = (s3 - s1) - s2;
      if (r < g.m && c < g.n) Cb[(long long)r * g.n + c] = cmake(sr, si);
    }
}

template <int BM, int BN, int STAGES, int NWARPS, bool A_KC, bool B_KC>
static void launch_gemm_l(const Arena& a, GemmArgs g) {
  constexpr int TA = (BM * LDK > BK * (BM + 2)) ? BM * LDK : BK * (BM + 2);
  constexpr int TB = (BN * LDK > BK * (BN + 2)) ? BN * LDK : BK * (BN + 2);
  constexpr size_t smem = sizeof(double2) * (size_t)STAGES * (TA + TB);
  const unsigned tn = (unsigned)((g.n + BN - 1) / BN), tm = (unsigned)((g.m + BM - 1) / BM);
  g.rows_on_x = tm > tn;
  dim3 grid(g.rows_on_x ? tm : tn, g.rows_on_x ? tn : tm, (unsigned)(a.nb * g.ksplit));
  zgemm_dmma_kernel<BM, BN, STAGES, NWARPS, A_KC, B_KC><<<grid, 32 * NWARPS, smem, a.stream>>>(a.base, a.chain_stride, g);
  ++*a.launches;
}

// operand layouts are template parameters (a kernel that takes them at run time carries every fragment-load variant
// in its unrolled loops: ~56 KB of code, instruction-cache misses were 20 % of the stall samples of the small products)
template <int BM, int BN, int STAGES, int NWARPS>
static void launch_gemm(const Arena& a, const GemmArgs& g) {
  const bool a_kc = (g.opA == OP_N || g.opA == OP_J), b_kc = (g.opB == OP_T || g.opB == OP_C);
  if (a_kc && b_kc) launch_gemm_l<BM, BN, STAGES, NWARPS, true, true>(a, g);
  else if (a_kc) launch_gemm_l<BM, BN, STAGES, NWARPS, true, false>(a, g);
  else if (b_kc) launch_gemm_l<BM, BN, STAGES, NWARPS, false, true>(a, g);
  else launch_gemm_l<BM, BN, STAGES, NWARPS, false, false>(a, g);
}

void gemm_splitk(const Arena& a, int64_t C, int64_t A, int64_t B, int64_t m, int64_t n, int64_t k, int opA, int opB, int ksplit) {
  if (m == 0 || n == 0) return;
  if (a.gemm_flops && a.depth == 0) *a.gemm_flops += 6.0 * (double)m * (double)n * (double)k * a.nb;   // (bodies of conditional nodes not counted)
  static const bool ktime = getenv("KBP_KTIME") != nullptr;
  static int kt_next = 0;                                     // (probe runs are single-threaded at capture time)
  GemmArgs g{C, A, B, (int)m, (int)n, (int)k, opA, opB, ksplit < 1 ? 1 : ksplit, 0, 0, a.scratch, a.scratch_stride, a.counters_dev, a.mask, a.mask_want,
             (ktime && m * n * k >= 8 * 1024 * 1024) ? (kt_next++ % GEMM_KT_SLOTS) : -1};
  if (ksplit == 0) {
    // automatic: a small product is bound by how many warps (16x8 accumulator tiles) it offers to the 592 sub-partitions;
    // split k (fused, deterministic reduction) until there are enough, keeping >= 4 slabs per split
    const int64_t tiles16 = ((n + 15) / 16) * ((m + 15) / 16);
    const int64_t warps = 2 * tiles16 * a.nb;
    const int64_t slabs = (k + BK - 1) / BK;
    int ks = 1;
    if (warps < 600 && slabs >= 8 && tiles16 <= GEMM_MAX_TILES && a.scratch != nullptr) {
      ks = (int)((GEMM_WARPS_TARGET + warps - 1) / warps);
      if (ks > slabs / 4) ks = (int)(slabs / 4);
      if (ks > 16) ks = 16;
      while (ks > 1 && (int64_t)ks * m * n > a.scratch_stride) --ks;
    }
    g.ksplit = ks < 1 ? 1 : ks;
    g.fused = g.ksplit > 1;
  }
  // FP64 DMMA runs at 64 FMA/clk/SM: a 32x32 tile needs ~1000 cycles per 16-deep k-slab, so a product that covers only a
  // few dozen tiles is bound by the handful of SMs it occupies.  Pick the largest tile that still spreads over the machine.
  const int64_t ctas64 = ((n + 63) / 64) * ((m + 63) / 64) * a.nb * g.ksplit;
  const int64_t ctas32 = ((n + 31) / 32) * ((m + 31) / 32) * a.nb * g.ksplit;
  // The 16 x 16 tile runs 3 stages: measured, 3 stages (30 KB, 7 CTAs per SM) beat 4 on every shape of tools/gemm_bench.py d4.
  if (g.fused || ctas32 < 96) launch_gemm<16, 16, 3, 2>(a, g);
  else if (ctas64 >= 96) launch_gemm<64, 64, 3, 8>(a, g);
  else launch_gemm<32, 32, 4, 8>(a, g);
}

template <int BM, int BN, int STAGES, int NWARPS>
static void gemm_attr() {
  constexpr int TA = (BM * LDK > BK * (BM + 2)) ? BM * LDK : BK * (BM + 2);
  constexpr int TB = (BN * LDK > BK * (BN + 2)) ? BN * LDK : BK * (BN + 2);
  constexpr size_t smem = sizeof(double2) * (size_t)STAGES * (TA + TB);
  cudaFuncSetAttribute(zgemm_dmma_kernel<BM, BN, STAGES, NWARPS, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaFuncSetAttribute(zgemm_dmma_kernel<BM, BN, STAGES, NWARPS, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaFuncSetAttribute(zgemm_dmma_kernel<BM, BN, STAGES, NWARPS, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaFuncSetAttribute(zgemm_dmma_kernel<BM, BN, STAGES, NWARPS, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

void gemm_ktime_report(const char* tag) {
  static std::vector<unsigned long long> t0(GEMM_KT_SLOTS), t1(GEMM_KT_SLOTS);
  cudaMemcpyFromSymbol(t0.data(), g_gemm_t0, sizeof(unsigned long long) * GEMM_KT_SLOTS);
  cudaMemcpyFromSymbol(t1.data(), g_gemm_t1, sizeof(unsigned long long) * GEMM_KT_SLOTS);
  double sum = 0;
  long long n = 0;
  for (int i = 0; i < GEMM_KT_SLOTS; ++i)
    if (t1[i] > t0[i] && t0[i] != ~0ull) { sum += (double)(t1[i] - t0[i]); ++n; }
  if (n) fprintf(stderr, "[kbp ktime] %s: %lld large GEMM launches (last replay), %.2f us each from first CTA start to last CTA main loop end\n", tag, n, 1e-3 * sum / n);
  std::fill(t0.begin(), t0.end(), ~0ull);
  std::fill(t1.begin(), t1.end(), 0ull);
  cudaMemcpyToSymbol(g_gemm_t0, t0.data(), sizeof(unsigned long long) * GEMM_KT_SLOTS);
  cudaMemcpyToSymbol(g_gemm_t1, t1.data(), sizeof(unsigned long long) * GEMM_KT_SLOTS);
}

void init_gemm_attributes() {
  gemm_attr<16, 16, 3, 2>();
  gemm_attr<32, 32, 4, 8>();
  gemm_attr<64, 64, 3, 8>();
}

void gemm(const Arena& a, int64_t C, int64_t A, int64_t B, int64_t m, int64_t n, int64_t k, int opA, int opB) {
  gemm_splitk(a, C, A, B, m, n, k, opA, opB, 0);
}

}  // namespace kbp
