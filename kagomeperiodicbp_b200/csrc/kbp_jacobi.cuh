// One-sided (Hestenes) Jacobi building blocks of the one-CTA SVD: the round-robin pair schedule, the lane-group reduction of a
// pair's Gram sums, the rotation and its application to a row pair held in registers.  Used by the truncated SVD of small
// matrices (k_svd_small.cu) and by the simple-update kernel (k_su.cu).
#pragma once
#include "kbp_common.cuh"

namespace kbp {

constexpr double SMALL_TOL = 1e-14;

// Round-robin tournament on pp (even) players: in step r, slot 0 pairs player pp-1 with r, slot t > 0 pairs (r + t) mod (pp-1)
// with (r - t) mod (pp-1).  The two residues are carried from step to step (no integer division in the step loop).
struct PairWalk {
  int ra, rb, m1, slot;
  __device__ __forceinline__ void start(int pp, int slot_) { m1 = pp - 1; slot = slot_; ra = slot_; rb = slot_ == 0 ? 0 : m1 - slot_; }
  __device__ __forceinline__ void get(int step, int& i, int& j) const {
    if (slot == 0) { i = step; j = m1; }
    else { i = ra < rb ? ra : rb; j = ra < rb ? rb : ra; }
  }
  __device__ __forceinline__ void next() { ra = ra + 1 == m1 ? 0 : ra + 1; rb = rb + 1 == m1 ? 0 : rb + 1; }
};

struct __align__(16) PairSums { double a, b, cr, ci; };

// Sum (a, b, cr, ci) over the G lanes of a group and hand all four totals to every lane.  Shuffles are the scarce resource
// here (one warp-shuffle per 4 cycles per SM sub-partition, two per double), so the butterfly is TRANSPOSED: the first two
// stages halve the number of values a lane carries (4 -> 2 -> 1) while doubling what each covers, the remaining stages
// reduce that single value: 4 + log2(G/4) double-shuffles instead of 4 log2(G).  The four owners then publish the totals
// through a 32-byte shared-memory record of the pair, which every lane reads back (broadcast loads).
template <int G>
__device__ __forceinline__ double group_reduce4(double a, double b, double cr, double ci, int gl, unsigned gmask) {
  static_assert(G >= 4, "group of at least 4 lanes");
  const bool b0 = gl & 1, b1 = gl & 2;
  double k0 = b0 ? cr : a, k1 = b0 ? ci : b;                       // even lanes keep (a, b), odd lanes keep (cr, ci)
  k0 += __shfl_xor_sync(gmask, b0 ? a : cr, 1);
  k1 += __shfl_xor_sync(gmask, b0 ? b : ci, 1);
  double mine = b1 ? k1 : k0;                                      // (b1, b0) = 00: a   01: cr   10: b   11: ci
  mine += __shfl_xor_sync(gmask, b1 ? k0 : k1, 2);
#pragma unroll
  for (int o = 4; o < G; o <<= 1) mine += __shfl_xor_sync(gmask, mine, o);
  return mine;
}
// position of lane gl's total inside PairSums {a, b, cr, ci}
__device__ __forceinline__ int owner_pos(int gl) { return ((gl & 1) << 1) | ((gl >> 1) & 1); }

// The rotation that orthogonalises rows x_i, x_j with Gram entries a = |x_i|^2, b = |x_j|^2, c = <x_i, x_j> = cr + i ci:
// x_j' = e x_j with e = c/|c| makes the inner product real, then a real rotation by theta, tan(2 theta) = 2|c| / (a - b),
// |theta| <= pi/4.  With h = (a-b)^2 + 4|c|^2:  cos^2(theta) = (1 + |a-b|/sqrt(h)) / 2,  sin(theta) = |c| / (sqrt(h) cos(theta)):
// two levels of special functions (rsqrt(|c|^2) || rsqrt(h), then rsqrt(cos^2)) and no division; products only, so a tiny
// |c| keeps its relative accuracy.  Returns false when the pair is already orthogonal to tolerance (or a row is dead).
// `big` is raised when cos^2 of the pair's angle exceeded SMALL_TOL (the sweep-level convergence test).
struct Rotation { double cs, sn, er, ei; bool swap; };
__device__ __forceinline__ bool make_rotation(double a, double b, double cr, double ci, double floor2, bool& big, Rotation& R) {
  const double r2 = fma(cr, cr, ci * ci), ab = a * b;
  if (!(a > floor2 && b > floor2 && r2 > (SMALL_TOL * SMALL_TOL) * ab)) return false;
  big = big || r2 > SMALL_TOL * ab;
  const double d = a - b;
  const double h = fma(d, d, 4.0 * r2);
  const double ri = rsqrt(r2), rh = rsqrt(h);
  const double x = fma(0.5 * fabs(d), rh, 0.5);
  const double rs = rsqrt(x);
  const double sn = (r2 * ri) * rh * rs;
  R.cs = x * rs;
  R.sn = d < 0.0 ? -sn : sn;
  R.er = cr * ri;
  R.ei = ci * ri;
  R.swap = d < 0.0;                                  // keep the larger row first (de Rijk)
  return true;
}

// rotate one row pair with both rows held in registers between the Gram sums and the update (CPL columns per lane)
template <int CPL, int G>
__device__ __forceinline__ void jacobi_pair_cached(cplx* __restrict__ xi, cplx* __restrict__ xj, int q, int qx, int gl, unsigned gmask,
                                                   double floor2, bool& big, PairSums* __restrict__ rec) {
  cplx u[CPL], v[CPL];
  double a = 0.0, b = 0.0, cr = 0.0, ci = 0.0;
#pragma unroll
  for (int k = 0; k < CPL; ++k) {
    const int c = gl + k * G;
    u[k] = c < q ? xi[c] : cmake(0.0, 0.0);
    v[k] = c < q ? xj[c] : cmake(0.0, 0.0);
    if (c < qx) {                                  // Gram sums over the data columns only (not the accumulated rotations)
      a = fma(u[k].x, u[k].x, fma(u[k].y, u[k].y, a));
      b = fma(v[k].x, v[k].x, fma(v[k].y, v[k].y, b));
      cr = fma(u[k].x, v[k].x, fma(u[k].y, v[k].y, cr));          // u conj(v)
      ci = fma(u[k].y, v[k].x, fma(-u[k].x, v[k].y, ci));
    }
  }
  const double mine = group_reduce4<G>(a, b, cr, ci, gl, gmask);
  if (gl < 4) reinterpret_cast<double*>(rec)[owner_pos(gl)] = mine;
  __syncwarp(gmask);
  const PairSums tot = *rec;
  Rotation R;
  if (!make_rotation(tot.a, tot.b, tot.cr, tot.ci, floor2, big, R)) return;
#pragma unroll
  for (int k = 0; k < CPL; ++k) {
    const int c = gl + k * G;
    if (c < q) {
      const double vr = R.er * v[k].x - R.ei * v[k].y, vi = R.er * v[k].y + R.ei * v[k].x;     // e x_j
      const cplx yi = make_double2(fma(R.cs, u[k].x, R.sn * vr), fma(R.cs, u[k].y, R.sn * vi));
      const cplx yj = make_double2(fma(R.cs, vr, -R.sn * u[k].x), fma(R.cs, vi, -R.sn * u[k].y));
      xi[c] = R.swap ? yj : yi;
      xj[c] = R.swap ? yi : yj;
    }
  }
}

}  // namespace kbp
