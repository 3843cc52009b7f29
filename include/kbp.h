/* kbp.h -- C ABI of the B200 block-BP engine (libkbp.so).
 *
 * Plain pointers and sizes only; no torch / C++ types.  The library executes *tensor programs*:
 * flat int64 op streams over numbered complex128 buffers in a device arena that holds `nb`
 * independent chains (block sides x ensemble members) side by side.  The Python host
 * (kagomeperiodicbp_b200/) compiles the reference's call
 *
 *     bubblecon(T_list, edges_list, angles_list, bubble_angle, swallow_order, D_trunc, ...,
 *               ket_tensors, separate_exp, compression)          src/libs/bubblecon.py:2465-2468
 *
 * (its only live call site is src/algo/contract_tensor_network.py:193-205) and the per-message
 * epilogue of one BP iteration (_fix_messages / _compute_error / _message_damping,
 * src/algo/belief_propagation.py:113-117, 44-56, 59-87) into such a program; the ops are the
 * reference's numerical primitives:
 *
 *   KBP_OP_GEMM / KBP_OP_PERMUTE   numpy.tensordot / transpose in swallow_ket_T, swallow_T, merge_T
 *                                  (src/libs/bubblecon.py:1855-2172, 2180-2453, 994-1184)
 *   KBP_OP_QR                      numpy.linalg.qr in mps.left_canonical_QR, and (on the conjugate
 *                                  transpose) scipy.linalg.rq in mps.right_canonical
 *                                  (src/libs/bmpslib.py:553-595, 775-806)
 *   KBP_OP_SVD                     _perf_svd + truncation + S/|S| in mps.right_canonical
 *                                  (src/libs/bmpslib.py:733-772, 2873-2885)
 *   KBP_OP_NORMALIZE               mps.update_A0_norm (src/libs/bmpslib.py:359-375); the (mantissa, exp10)
 *                                  pair is kept as one natural-log slot per chain
 *   KBP_OP_EMBED / KBP_OP_ZERO     add_two_MPSs block placement (src/libs/bmpslib.py:2781-2864)
 *   KBP_OP_NONFINITE               the NaN/Inf guard of right_canonical (src/libs/bmpslib.py:711-717),
 *                                  surfaced as a flag instead of exit(1)
 *
 * Error behaviour: every entry point returns 0 on success, a negative KBP_E_* code otherwise;
 * kbp_last_error() gives the text.  The reference prints and calls exit(1) in these places
 * (src/libs/bubblecon.py:2921-2949, src/libs/bmpslib.py:711-717, 880-883); the Python shim raises
 * BubbleConError instead.
 */
#ifndef KBP_H
#define KBP_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct kbp_ctx kbp_ctx;

enum { KBP_OK = 0, KBP_E_CUDA = -1, KBP_E_ARG = -2, KBP_E_PROGRAM = -3, KBP_E_SVD_NOCONV = -4, KBP_E_NONFINITE = -5 };

enum {
  KBP_OP_PERMUTE = 1,        /* dst, src, conj, ndim, dims_src[ndim], perm[ndim] */
  KBP_OP_GEMM = 2,           /* C, A, B, m, n, k, opA, opB      op: 0 N, 1 T, 2 C (conj-transpose), 3 J (conj) */
  KBP_OP_QR = 3,             /* A, Q, R, work, m, n */
  KBP_OP_SVD = 4,            /* A, US, Vh, work, m, n, keep, nr_bulk, slot_lognorm, slot_trunc, reserved (-1) */
  KBP_OP_NORMALIZE = 5,      /* buf, n, slot_lognorm */
  KBP_OP_EMBED = 6,          /* dst, src, alpha_re(bits), alpha_im(bits), d0, d1, d2, s0, s1, s2, sign_slot */
  KBP_OP_ZERO = 7,           /* dst, n */
  KBP_OP_SCALAR_TO_SLOT = 8, /* buf, slot_re, slot_im */
  KBP_OP_NONFINITE = 9,      /* buf, n, slot */
  KBP_OP_EYE = 10,           /* dst, rows, cols : dst = identity (reshaped-identity MPS sites, src/libs/bubblecon.py:345-382) */
  KBP_OP_SU = 11             /* G_A, G_B, G_C, lambda, gate, rdm, d, D, max_steps, tol(bits), slot_steps, slot_delta, slot_nonfinite,
                                then 6 x (site_i, leg_i, site_j, leg_j):  simple update of the Kagome unit cell (Gamma [d, D, D, D, D]
                                x 3 and lambda 6 x D updated in place, gate d^4 in the layout g[i', i, j', j], rdm 6 x d^4 written),
                                one CTA per chain, up to max_steps Trotter steps, a chain stops when its step delta < tol; d = 2,
                                2 <= D <= 6 */
};

/* lifetime */
int kbp_create(int device, kbp_ctx** out);
void kbp_destroy(kbp_ctx* ctx);
const char* kbp_last_error(const kbp_ctx* ctx);
int kbp_device_count(void);

/* arena: nb chains x chain_elems complex128 elements, plus nb x n_slots doubles of scalar slots (zeroed).
 * The LAST slot of every chain is reserved by the engine: it counts truncations whose Jacobi iteration did not
 * converge (the asynchronous counterpart of the KBP_E_SVD_NOCONV return code). */
int kbp_reserve(kbp_ctx* ctx, int64_t chain_elems, int nb, int n_slots);

/* host <-> device.  `host` holds interleaved complex128.  chain = -1: `host` is [nb][n_elems], one row per chain. */
int kbp_upload(kbp_ctx* ctx, int chain, int64_t offset, const void* host, int64_t n_elems);
int kbp_download(kbp_ctx* ctx, int chain, int64_t offset, void* host, int64_t n_elems);
int kbp_broadcast(kbp_ctx* ctx, int64_t offset, const void* host, int64_t n_elems);   /* same data to every chain */
int kbp_slots_read(kbp_ctx* ctx, double* host);      /* nb * n_slots doubles */
int kbp_slots_zero(kbp_ctx* ctx);

/* run a tensor program on all chains.  From its second run on a program executes as ONE CUDA graph launch: the call is
 * asynchronous and no decision is taken on the host (the data-dependent loops of the truncated SVDs are conditional graph
 * nodes driven by device-side decision kernels).  The first run of a program, and every run when graphs are disabled
 * (KBP_GRAPHS=0, under Nsight Compute, with per-op profiling on), is host-driven: plain launches, one small read-back per
 * SVD decision.  kbp_graph_ready tells which of the two the next kbp_run of this program will be (1 = graph launch). */
int kbp_run(kbp_ctx* ctx, const int64_t* words, int64_t n_words);
int kbp_graph_ready(kbp_ctx* ctx, const int64_t* words, int64_t n_words);
/* programs shorter than min_words are never captured (default 256); capture_first != 0: capture at first sight (default: second) */
int kbp_graph_policy(kbp_ctx* ctx, int64_t min_words, int capture_first);
int kbp_sync(kbp_ctx* ctx);
/* SPECULATIVE program graphs (opt-in: KBP_SPECULATE=1 or kbp_set_speculation(ctx, 1)).  A captured program gives each truncated
 * SVD whose host-driven run was settled by the subspace iteration a FIXED schedule (the iterations it needed + one) and no
 * WHILE / IF node.  Every truncation still runs its acceptance test; a miss raises a sticky device flag.  Protocol: after the
 * program (kbp_run) and before using anything it wrote, call kbp_spec_failed (waits for the stream); if it returns 1, call
 * kbp_run_relearn with the same words -- inputs are never overwritten by a program, so they are still in place -- which runs
 * the program host-driven with every data-dependent loop and exact fallback, records the new schedule and drops the stale
 * graph.  kbp_spec_counters: out2[0] speculative graph launches, [1] failed ones.  Measured on the B200 (six side programs of
 * the D = 4, N = 6 block side by side): 648 ms per BP iteration against 672 ms with the conditional nodes -- and a schedule
 * learned from staged rounds misses its test now and then even on unchanged inputs, which costs a host-driven rerun; hence
 * off by default.  With speculation off kbp_spec_failed always returns 0. */
int kbp_spec_failed(kbp_ctx* ctx);
int kbp_run_relearn(kbp_ctx* ctx, const int64_t* words, int64_t n_words);
int kbp_set_speculation(kbp_ctx* ctx, int on);
/* developer probe (KBP_KTIME=1 in the environment): print and reset the in-kernel wall time of the Cholesky CTAs */
int kbp_ktime_report(kbp_ctx* ctx, const char* tag);
int kbp_spec_counters(const kbp_ctx* ctx, int64_t* out2);

/* device addresses of the arena ([nb][chain_elems] complex128), of the slot table ([nb][n_slots] doubles) and the CUDA stream
 * handle of the context, for zero-copy exchange of block messages between the arenas of different GPUs (NCCL all-gather in
 * kagomeperiodicbp_b200/parallel.py).  Valid until the next kbp_reserve that grows the arena. */
uint64_t kbp_arena_ptr(const kbp_ctx* ctx);
uint64_t kbp_slots_ptr(const kbp_ctx* ctx);
uint64_t kbp_stream_ptr(const kbp_ctx* ctx);
int64_t kbp_chain_elems(const kbp_ctx* ctx);

/* workspace sizes (complex128 elements) needed by KBP_OP_SVD / KBP_OP_QR */
int64_t kbp_svd_work_elems(int64_t m, int64_t n);
int64_t kbp_qr_work_elems(int64_t m, int64_t n);
/* reserved (size of a persistent per-op buffer; always 0: KBP_OP_SVD keeps no state between runs) */
int64_t kbp_svd_warm_elems(int64_t m, int64_t n, int64_t keep);

/* instrumentation: kernels launched so far; device timing of a region on the context's stream */
int64_t kbp_launch_count(const kbp_ctx* ctx);
/* real floating-point operations EXECUTED so far by the ZGEMM launches of this context (6 m n k per complex product: three real
 * DMMA products, 3M form); launches inside the bodies of conditional graph nodes (rounds beyond the learned schedule) are not
 * counted.  Against the algorithmic count of the reference's full SVDs this is what the tensor pipe really does. */
double kbp_gemm_flops(const kbp_ctx* ctx);
int64_t kbp_svd_sweeps(kbp_ctx* ctx);                 /* total block-Jacobi sweeps + subspace iterations so far (synchronises) */
/* how the truncations were executed so far (synchronises; [2..7] are counted on the device by the decision kernels):
 * out8[0] Householder reduction + in-shared-memory Jacobi, [1] in-shared-memory Jacobi, [2] accepted from subspace iteration,
 * [3] handed by the subspace iteration to the exact path, [4] exact (block-Jacobi) runs, [5] subspace iterations in total,
 * [6] block-Jacobi sweeps, [7] truncations that did not converge */
int kbp_svd_counters(kbp_ctx* ctx, int64_t* out8);
/* out4[0] graph launches so far, [1] programs captured, [2] graphs alive, [3] programs whose capture failed */
int kbp_graph_counters(const kbp_ctx* ctx, int64_t* out4);
int kbp_timer_start(kbp_ctx* ctx);
int kbp_timer_stop_ms(kbp_ctx* ctx, double* ms);       /* synchronises */
/* per-opcode device time: when enabled, kbp_run brackets every op with CUDA events on the context's stream;
 * kbp_profile_read synchronises and returns accumulated milliseconds and op counts indexed by opcode (16 entries) */
int kbp_profile_enable(kbp_ctx* ctx, int on);
int kbp_profile_read(kbp_ctx* ctx, double* ms16, int64_t* count16);

#ifdef __cplusplus
}
#endif
#endif
