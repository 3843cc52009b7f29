// Host-side launchers of the batched complex128 kernels.  Every launcher works on `nb` independent
// chains laid out in one arena: chain c's copy of a buffer lives at  base + c*chain_stride + offset
// (complex128 elements).  All launches are asynchronous on `stream`; none synchronises except
// svd_truncate (one flag read per Jacobi sweep).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <unordered_map>

namespace kbp {

// Device-side control block of the truncation in flight on a context's stream.  Every data-dependent decision of a truncated
// SVD (accept the subspace found / iterate further / hand the matrix to the exact Jacobi path; another Jacobi sweep or not) is
// taken ON THE DEVICE by a one-thread kernel that writes this block and, when the program runs as a CUDA graph, sets the
// condition of the WHILE / IF node that holds the optional work.  The host-driven mode (first run of a program, profilers)
// reads the same block back instead.  Followed in memory by `int state[nb]`.
struct SvdCtl {
  int round;               // subspace rounds (Rayleigh-Ritz + check) done by the op in flight
  int any_run;             // some chain wants another round
  int any_exact;           // some chain needs the exact path
  int sweeps;              // block-Jacobi sweeps done
  int any_sweep;           // some chain has not converged yet
  int pad[3];
  long long counters[8];   // [2] truncations accepted from subspace iteration, [3] handed to the exact path, [4] exact-path runs,
                           // [5] subspace iterations, [6] block-Jacobi sweeps, [7] truncations that did not converge
};
enum { CHAIN_RUNNING = 0, CHAIN_ACCEPTED = 1, CHAIN_EXACT = 2 };

// partial sums of the subspace-SVD check kernels: [nb][TSVD_NPART][TSVD_PART_STRIDE] doubles behind the 6 per-chain scalars
// of Arena::svd_off (TSVD_PART_STRIDE: keep <= 128 row sums + 2 norms); 3 more doubles per chain follow (block-Jacobi flags)
constexpr int TSVD_NPART = 128;
constexpr int TSVD_PART_STRIDE = 160;
constexpr int SVD_OFF_DOUBLES_PER_CHAIN = 6 + TSVD_NPART * TSVD_PART_STRIDE + 3;

struct Arena {
  double2* base;          // nb * chain_stride complex128 elements
  int64_t chain_stride;   // elements per chain
  double* slots;          // nb * n_slots doubles (log-norms, truncation errors, flags)
  int n_slots;
  int nb;
  cudaStream_t stream;
  cudaEvent_t block_event;  // non-null: host waits block on this event (yield the core) instead of spinning in cudaStreamSynchronize
  double2* scratch;       // split-K partial tiles: [nb][scratch_stride] complex128 (may be null)
  int64_t scratch_stride;
  int* counters_dev;      // split-K tile semaphores: [nb][4096] ints, zero between launches
  int64_t* launches;      // host counter of kernel launches
  double* gemm_flops;     // host counter (may be null): real flops the ZGEMM launches execute (6 m n k per complex product: 3M form)
  int64_t* counters;      // host counters [8]: see svd_truncate
  SvdCtl* ctl;            // device control block (+ state[nb]) of the truncation in flight, and its pinned host mirror
  SvdCtl* ctl_host;
  int* chain_state;       // device: [nb] CHAIN_* of the truncation in flight
  // per-chain predicate of the launches issued through this Arena: a kernel works on chain c iff mask == nullptr or
  // mask[c] == mask_want (chains of an ensemble converge after different numbers of rounds)
  const int* mask;
  int mask_want;
  // whole-program stream capture in progress: data-dependent loops become conditional graph nodes whose bodies are captured
  // on body_stream[depth]; conditional handles are created on top_graph
  // rounds the subspace iteration of each SVD op needed in the host-driven run of its program (key: program hash ^ word
  // index of the op): the captured graph gives such an op its iterations up front and does the Rayleigh-Ritz step once
  std::unordered_map<unsigned long long, int>* tsvd_rounds;
  unsigned long long op_key;
  bool capture;
  cudaGraph_t top_graph;
  cudaStream_t body_stream[2];
  int depth;
  // scratch for the Jacobi SVD convergence flags (device, nb doubles x 2) and its pinned host mirror
  double* svd_off;        // device: [6 + 32*160][nb]  (Jacobi: off current / previous sweep, ||A||_F^2; subspace: pivot, residual,
                          // ratio, discarded fraction, norms, partial sums of the check kernels)
  double* svd_off_host;   // pinned host mirror: [4][nb]
};

// host wait for everything queued on the arena's stream.  With several ranks x six launch threads per node the default
// spin-wait oversubscribes the host cores; a blocking event wait costs a few tens of microseconds once or twice per SVD.
inline cudaError_t stream_wait(const Arena& a) {
  if (!a.block_event) return cudaStreamSynchronize(a.stream);
  cudaError_t e = cudaEventRecord(a.block_event, a.stream);
  if (e != cudaSuccess) return e;
  return cudaEventSynchronize(a.block_event);
}

// CUDA graphs (whole programs in kbp_run, data-dependent loops as conditional nodes): on by default,
// KBP_GRAPHS=0/1 decides explicitly.  Under Nsight Compute they are off unless asked for: on this toolchain the tool aborts
// on stream capture from several threads with cluster launches, and a kernel-by-kernel profile wants plain launches anyway.
inline bool graphs_enabled() {
  static const bool on = [] {
    if (const char* e = getenv("KBP_GRAPHS")) return atoi(e) != 0;
    if (getenv("NV_COMPUTE_PROFILER_PERFWORKS_DIR") || getenv("NV_NSIGHT_INJECTION_PORT_BASE") || getenv("KBP_TSVD_PROF")) return false;
    return true;
  }();
  return on;
}

enum GemmOp { OP_N = 0, OP_T = 1, OP_C = 2, OP_J = 3 };   // as-is, transpose, conj-transpose, conj

// dst[contiguous, shape dims_src[perm]] = (conj?) src[contiguous, shape dims_src] transposed by perm
void permute(const Arena& a, int64_t dst, int64_t src, int conj, int ndim, const int64_t* dims_src, const int64_t* perm);
// C(m x n) = opA(A) * opB(B), row-major, inner dimension k
void gemm(const Arena& a, int64_t C, int64_t A, int64_t B, int64_t m, int64_t n, int64_t k, int opA, int opB);
// A(m x n) = Q(m x r) R(r x n), r = min(m, n), Q^H Q = I.  work: m*n + n elements
void qr(const Arena& a, int64_t A, int64_t Q, int64_t R, int64_t work, int64_t m, int64_t n);
// the same on a thread-block cluster with the matrix in distributed shared memory; false: shape not handled, nothing launched
bool qr_cluster(const Arena& a, int64_t A, int64_t Q, int64_t R, int64_t m, int64_t n);
// rank-`keep` truncated SVD of A(m x n):  US(m x keep) = U_k diag(s_k) [ / ||A||_F if nr_bulk ],  Vh(keep x n).
// slot_lognorm += ln ||A||_F (if nr_bulk); slot_trunc += sqrt(sum_discarded s^2 / sum s^2).
// work: see svd_work_elems().  Returns the number of Jacobi sweeps used (max over chains), <0 on failure.
int svd_truncate(const Arena& a, int64_t A, int64_t US, int64_t Vh, int64_t work, int64_t m, int64_t n, int64_t keep,
                 int nr_bulk, int slot_lognorm, int slot_trunc);
void ktime_report(const char* tag);
// opt-in of every kernel to > 48 KB of dynamic shared memory on the CURRENT device (called once per device by kbp_create)
void init_device_attributes();
// conditional node (WHILE or IF) appended to the capture in progress on a.stream; the returned Arena launches into its body.
// end_body() closes the body capture.  Both return false on a CUDA error.
bool begin_cond_body(const Arena& a, cudaGraphConditionalHandle h, bool is_while, Arena* body);
bool end_body(const Arena& body);
cudaGraphConditionalHandle new_cond_handle(const Arena& a);
bool svd_small_fits(int64_t m, int64_t n);
// ksplit >= 1: C partial sums side by side (C + s*m*n, s < ksplit), each over a contiguous range of k;  ksplit == 0: automatic
// fused split (partials in the scratch area, last CTA per tile reduces) -- what gemm() does
void gemm_splitk(const Arena& a, int64_t C, int64_t A, int64_t B, int64_t m, int64_t n, int64_t k, int opA, int opB, int ksplit);
int64_t svd_work_elems(int64_t m, int64_t n);
// buf /= ||buf||_F ; slot += ln ||buf||_F
void normalize(const Arena& a, int64_t buf, int64_t n, int slot_lognorm);
// dst[dst_off + i*s0 + j*s1 + k*s2] = alpha * src[(i*d1 + j)*d2 + k]; if sign_slot >= 0, alpha *= sign(slots[sign_slot]) (>0 -> +1, else -1)
void embed(const Arena& a, int64_t dst, int64_t src, double alpha_re, double alpha_im, int64_t d0, int64_t d1, int64_t d2,
           int64_t s0, int64_t s1, int64_t s2, int sign_slot);
void zero(const Arena& a, int64_t dst, int64_t n);
void eye(const Arena& a, int64_t dst, int64_t rows, int64_t cols);
// slots[slot_re], slots[slot_im] = buf[0]   (copy a device scalar into the slot table)
void scalar_to_slot(const Arena& a, int64_t buf, int slot_re, int slot_im);
// NaN/Inf guard: slots[slot] += (number of non-finite entries in buf)
void count_nonfinite(const Arena& a, int64_t buf, int64_t n, int slot);
// simple update of the three-site Kagome unit cell, one CTA per chain (k_su.cu); w = the 37 argument words of KBP_OP_SU
bool su_supported(int d, int D);
void simple_update(const Arena& a, const int64_t* w);

}  // namespace kbp
