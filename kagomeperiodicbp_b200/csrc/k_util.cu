// Layout / bookkeeping kernels: tensor permute (+conj), block embed (MPS addition), Frobenius
// normalisation with log-scale accumulation, NaN/Inf guard.  All HBM/L2-bound, coalesced on the
// write side, one grid row per chain.
#include "kbp_common.cuh"
#include "kbp_ops.cuh"

namespace kbp {

static inline int grid_for(int64_t n, int threads, int cap = 148 * 16) {
  int64_t g = (n + threads - 1) / threads;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

struct PermArgs {
  int ndim;
  int conj;
  long long total;
  long long ddim[8];     // destination dims
  long long sstride[8];  // source stride of each destination axis
};

__global__ void permute_kernel(cplx* __restrict__ base, long long chain_stride, long long dst, long long src, PermArgs p) {
  cplx* d = base + (long long)blockIdx.y * chain_stride + dst;
  const cplx* s = base + (long long)blockIdx.y * chain_stride + src;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < p.total; i += (long long)gridDim.x * blockDim.x) {
    long long rem = i, off = 0;
#pragma unroll 1
    for (int a = p.ndim - 1; a >= 0; --a) {
      long long c = rem % p.ddim[a];
      rem /= p.ddim[a];
      off += c * p.sstride[a];
    }
    cplx v = s[off];
    if (p.conj) v.y = -v.y;
    d[i] = v;
  }
}

void permute(const Arena& a, int64_t dst, int64_t src, int conj, int ndim, const int64_t* dims_src, const int64_t* perm) {
  PermArgs p;
  long long sstr[8];
  long long acc = 1;
  for (int i = ndim - 1; i >= 0; --i) { sstr[i] = acc; acc *= dims_src[i]; }
  // merge nothing, just map
  p.ndim = ndim;
  p.conj = conj;
  p.total = acc;
  for (int i = 0; i < ndim; ++i) { p.ddim[i] = dims_src[perm[i]]; p.sstride[i] = sstr[perm[i]]; }
  for (int i = ndim; i < 8; ++i) { p.ddim[i] = 1; p.sstride[i] = 0; }
  if (acc == 0) return;
  dim3 g(grid_for(acc, 256), a.nb);
  permute_kernel<<<g, 256, 0, a.stream>>>(a.base, a.chain_stride, dst, src, p);
  ++*a.launches;
}

__global__ void embed_kernel(cplx* __restrict__ base, long long chain_stride, const double* __restrict__ slots, int n_slots,
                             long long dst, long long src, cplx alpha, long long d0, long long d1, long long d2,
                             long long s0, long long s1, long long s2, int sign_slot) {
  cplx* d = base + (long long)blockIdx.y * chain_stride + dst;
  const cplx* s = base + (long long)blockIdx.y * chain_stride + src;
  if (sign_slot >= 0) {
    double sg = slots[(long long)blockIdx.y * n_slots + sign_slot] > 0 ? 1.0 : -1.0;
    alpha.x *= sg;
    alpha.y *= sg;
  }
  long long total = d0 * d1 * d2;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long k = i % d2, r = i / d2;
    long long j = r % d1, q = r / d1;
    d[q * s0 + j * s1 + k * s2] = cmul(alpha, s[i]);
  }
}

void embed(const Arena& a, int64_t dst, int64_t src, double ar, double ai, int64_t d0, int64_t d1, int64_t d2,
           int64_t s0, int64_t s1, int64_t s2, int sign_slot) {
  int64_t total = d0 * d1 * d2;
  if (total == 0) return;
  dim3 g(grid_for(total, 256), a.nb);
  embed_kernel<<<g, 256, 0, a.stream>>>(a.base, a.chain_stride, a.slots, a.n_slots, dst, src, cmake(ar, ai), d0, d1, d2, s0, s1, s2, sign_slot);
  ++*a.launches;
}

__global__ void zero_kernel(cplx* __restrict__ base, long long chain_stride, long long dst, long long n) {
  cplx* d = base + (long long)blockIdx.y * chain_stride + dst;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) d[i] = cmake(0.0, 0.0);
}

void zero(const Arena& a, int64_t dst, int64_t n) {
  if (n == 0) return;
  dim3 g(grid_for(n, 256), a.nb);
  zero_kernel<<<g, 256, 0, a.stream>>>(a.base, a.chain_stride, dst, n);
  ++*a.launches;
}

__global__ void eye_kernel(cplx* __restrict__ base, long long chain_stride, long long dst, long long rows, long long cols) {
  cplx* d = base + (long long)blockIdx.y * chain_stride + dst;
  const long long n = rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    d[i] = cmake((i / cols) == (i % cols) ? 1.0 : 0.0, 0.0);
}

void eye(const Arena& a, int64_t dst, int64_t rows, int64_t cols) {
  if (rows * cols == 0) return;
  dim3 g(grid_for(rows * cols, 256), a.nb);
  eye_kernel<<<g, 256, 0, a.stream>>>(a.base, a.chain_stride, dst, rows, cols);
  ++*a.launches;
}

// one CTA per chain: ||buf||_F by a block reduction (warp shuffles inside), then rescale in place.
__global__ void normalize_kernel(cplx* __restrict__ base, long long chain_stride, double* __restrict__ slots, int n_slots,
                                 long long buf, long long n, int slot) {
  __shared__ double red[34];
  cplx* d = base + (long long)blockIdx.x * chain_stride + buf;
  // two-pass scaled norm: max |x| first so the squares cannot overflow/underflow
  double mx = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) mx = fmax(mx, fmax(fabs(d[i].x), fabs(d[i].y)));
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x < 32) {
    double t = threadIdx.x < ((blockDim.x + 31) >> 5) ? red[threadIdx.x] : 0.0;
    t = warp_max(t);
    if (threadIdx.x == 0) red[33] = t;
  }
  __syncthreads();
  mx = red[33];
  if (!(mx > 0.0) || !isfinite(mx)) return;   // all-zero or non-finite: leave untouched
  double inv = 1.0 / mx, acc = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) {
    double x = d[i].x * inv, y = d[i].y * inv;
    acc = fma(x, x, fma(y, y, acc));
  }
  double nrm = mx * sqrt(block_sum(acc, red));
  double r = 1.0 / nrm;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) d[i] = cscale(d[i], r);
  if (threadIdx.x == 0 && slot >= 0) slots[(long long)blockIdx.x * n_slots + slot] += log(nrm);
}

void normalize(const Arena& a, int64_t buf, int64_t n, int slot) {
  if (n == 0) return;
  normalize_kernel<<<a.nb, 512, 0, a.stream>>>(a.base, a.chain_stride, a.slots, a.n_slots, buf, n, slot);
  ++*a.launches;
}

__global__ void scalar_to_slot_kernel(const cplx* __restrict__ base, long long chain_stride, double* __restrict__ slots, int n_slots,
                                      long long buf, int sre, int sim, int nb) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nb) return;
  cplx v = base[(long long)c * chain_stride + buf];
  if (sre >= 0) slots[(long long)c * n_slots + sre] = v.x;
  if (sim >= 0) slots[(long long)c * n_slots + sim] = v.y;
}

void scalar_to_slot(const Arena& a, int64_t buf, int sre, int sim) {
  scalar_to_slot_kernel<<<(a.nb + 63) / 64, 64, 0, a.stream>>>(a.base, a.chain_stride, a.slots, a.n_slots, buf, sre, sim, a.nb);
  ++*a.launches;
}

__global__ void nonfinite_kernel(const cplx* __restrict__ base, long long chain_stride, double* __restrict__ slots, int n_slots,
                                 long long buf, long long n, int slot) {
  __shared__ double red[34];
  const cplx* d = base + (long long)blockIdx.x * chain_stride + buf;
  double bad = 0.0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x)
    if (!isfinite(d[i].x) || !isfinite(d[i].y)) bad += 1.0;
  bad = block_sum(bad, red);
  if (threadIdx.x == 0 && bad > 0) slots[(long long)blockIdx.x * n_slots + slot] += bad;
}

void count_nonfinite(const Arena& a, int64_t buf, int64_t n, int slot) {
  if (n == 0) return;
  nonfinite_kernel<<<a.nb, 256, 0, a.stream>>>(a.base, a.chain_stride, a.slots, a.n_slots, buf, n, slot);
  ++*a.launches;
}

}  // namespace kbp

namespace kbp {
void init_gemm_attributes();
void init_qr_attributes();
void init_svd_attributes();
void init_svd_small_attributes();
void init_tsvd_attributes();
void init_su_attributes();
void init_device_attributes() {
  init_gemm_attributes();
  init_qr_attributes();
  init_svd_attributes();
  init_svd_small_attributes();
  init_tsvd_attributes();
  init_su_attributes();
}
}  // namespace kbp
