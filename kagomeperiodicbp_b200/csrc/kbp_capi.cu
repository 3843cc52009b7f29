// C ABI of libkbp.so (see include/kbp.h): context, device arena, transfers, tensor-program interpreter.
#include "../../include/kbp.h"

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>

#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "kbp_ops.cuh"

static const int64_t KBP_GEMM_SCRATCH = 1 << 20;   // complex128 elements per chain for split-K partial tiles (16 MB)

struct kbp_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  double2* arena = nullptr;
  int64_t chain_elems = 0;
  int nb = 0;
  double* slots = nullptr;
  int n_slots = 0;
  double2* scratch = nullptr;
  int* counters_dev = nullptr;
  double* svd_off = nullptr;
  double* svd_off_host = nullptr;
  int64_t launches = 0;
  double gemm_flops = 0;                 // real flops executed by the ZGEMM launches so far (3M form: 6 m n k each)
  int64_t counters[8] = {0};
  kbp::SvdCtl* ctl = nullptr;            // device control block of the truncation in flight, followed by int state[nb]
  kbp::SvdCtl* ctl_host = nullptr;       // pinned mirror (host-driven mode, counters)
  cudaStream_t body_stream[2] = {nullptr, nullptr};   // capture streams of conditional-node bodies
  struct GraphEntry { cudaGraphExec_t exec = nullptr; int seen = 0; int64_t launches = 0; int64_t dcount[8] = {0}; double flops = 0; bool bad = false; };
  std::unordered_map<uint64_t, GraphEntry> graphs;      // CUDA graphs of whole programs, keyed by a hash of the op stream
  std::unordered_map<unsigned long long, int> tsvd_rounds;
  int64_t graph_replays = 0;
  int64_t graph_captures = 0;
  int64_t graph_min_words = 256;         // shorter programs (one-off algebra of the ITE step) run as plain launches
  bool graph_first = false;              // capture a program the first time it is seen (default: the second)
  bool profile = false;
  struct Span { int op; cudaEvent_t a, b; };
  std::vector<Span> spans;
  double prof_ms[16] = {0};
  int64_t prof_n[16] = {0};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t block_event = nullptr;
  std::string err;
};

static int fail(kbp_ctx* c, int code, const std::string& msg) {
  if (c) c->err = msg;
  return code;
}

#define CU(c, call)                                                                                   \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess) return fail(c, KBP_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

static cudaError_t ctx_wait(kbp_ctx* c) {
  if (!c->block_event) return cudaStreamSynchronize(c->stream);
  cudaError_t e = cudaEventRecord(c->block_event, c->stream);
  if (e != cudaSuccess) return e;
  return cudaEventSynchronize(c->block_event);
}

extern "C" {

int kbp_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int kbp_create(int device, kbp_ctx** out) {
  if (!out) return KBP_E_ARG;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) return KBP_E_CUDA;     // no CPU fallback: the caller must fail loudly
  if (device < 0 || device >= n) return KBP_E_ARG;
  kbp_ctx* c = new kbp_ctx();
  c->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->body_stream[0], cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->body_stream[1], cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&c->ev0) != cudaSuccess || cudaEventCreate(&c->ev1) != cudaSuccess) {
    delete c;
    return KBP_E_CUDA;
  }
  {
    // the > 48 KB shared-memory opt-in is a per-device function attribute: set once for every device a context is made on
    static std::mutex mu;
    static bool done[64] = {false};
    std::lock_guard<std::mutex> lk(mu);
    if (device < 64 && !done[device]) { kbp::init_device_attributes(); done[device] = true; cudaGetLastError(); }
  }
  // blocking host waits on request (KBP_BLOCKING_SYNC=1): useful when many ranks share few host cores; measured on a
  // 4 x B200 / 32-core box the default spin wait is ~6 % faster, so it stays the default
  const char* bs = getenv("KBP_BLOCKING_SYNC");
  const bool blocking = bs && atoi(bs) != 0;
  if (blocking && cudaEventCreateWithFlags(&c->block_event, cudaEventBlockingSync | cudaEventDisableTiming) != cudaSuccess) c->block_event = nullptr;
  *out = c;
  return KBP_OK;
}

static void drop_graphs(kbp_ctx* c) {
  for (auto& kv : c->graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  c->graphs.clear();
}

static void fold_device_counters(kbp_ctx* c) {
  if (!c->ctl || !c->ctl_host) return;
  if (cudaMemcpyAsync(c->ctl_host, c->ctl, sizeof(kbp::SvdCtl), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) return;
  if (cudaStreamSynchronize(c->stream) != cudaSuccess) return;
  for (int k = 2; k < 8; ++k) c->counters[k] += c->ctl_host->counters[k];
  cudaMemsetAsync(reinterpret_cast<char*>(c->ctl) + offsetof(kbp::SvdCtl, counters), 0, sizeof(long long) * 8, c->stream);
}

static void free_arena(kbp_ctx* c) {
  fold_device_counters(c);
  drop_graphs(c);
  if (c->arena) cudaFree(c->arena);
  if (c->slots) cudaFree(c->slots);
  if (c->scratch) cudaFree(c->scratch);
  if (c->counters_dev) cudaFree(c->counters_dev);
  c->scratch = nullptr; c->counters_dev = nullptr;
  if (c->svd_off) cudaFree(c->svd_off);
  if (c->svd_off_host) cudaFreeHost(c->svd_off_host);
  if (c->ctl) cudaFree(c->ctl);
  if (c->ctl_host) cudaFreeHost(c->ctl_host);
  c->ctl = nullptr; c->ctl_host = nullptr;
  c->arena = nullptr; c->slots = nullptr; c->svd_off = nullptr; c->svd_off_host = nullptr;
  c->chain_elems = 0; c->nb = 0; c->n_slots = 0;
}

void kbp_destroy(kbp_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  free_arena(c);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  if (c->block_event) cudaEventDestroy(c->block_event);
  if (c->stream) cudaStreamDestroy(c->stream);
  for (int i = 0; i < 2; ++i)
    if (c->body_stream[i]) cudaStreamDestroy(c->body_stream[i]);
  delete c;
}

const char* kbp_last_error(const kbp_ctx* c) { return c ? c->err.c_str() : "null context"; }

int kbp_reserve(kbp_ctx* c, int64_t chain_elems, int nb, int n_slots) {
  if (!c || chain_elems <= 0 || nb <= 0 || n_slots <= 0) return fail(c, KBP_E_ARG, "kbp_reserve: bad argument");
  CU(c, cudaSetDevice(c->device));
  CU(c, ctx_wait(c));
  if (chain_elems > c->chain_elems || nb != c->nb || n_slots != c->n_slots) {
    free_arena(c);
    CU(c, cudaMalloc(&c->arena, sizeof(double2) * (size_t)chain_elems * nb));
    CU(c, cudaMalloc(&c->slots, sizeof(double) * (size_t)nb * n_slots));
    CU(c, cudaMalloc(&c->scratch, sizeof(double2) * (size_t)KBP_GEMM_SCRATCH * nb));
    CU(c, cudaMalloc(&c->counters_dev, sizeof(int) * (size_t)4096 * nb));
    CU(c, cudaMemsetAsync(c->counters_dev, 0, sizeof(int) * (size_t)4096 * nb, c->stream));
    CU(c, cudaMalloc(&c->svd_off, sizeof(double) * (size_t)kbp::SVD_OFF_DOUBLES_PER_CHAIN * nb));
    CU(c, cudaMallocHost(&c->svd_off_host, sizeof(double) * 4 * nb));
    CU(c, cudaMalloc(&c->ctl, sizeof(kbp::SvdCtl) + sizeof(int) * (size_t)nb));
    CU(c, cudaMemsetAsync(c->ctl, 0, sizeof(kbp::SvdCtl) + sizeof(int) * (size_t)nb, c->stream));
    CU(c, cudaMallocHost(&c->ctl_host, sizeof(kbp::SvdCtl)));
    memset(c->ctl_host, 0, sizeof(kbp::SvdCtl));
    c->chain_elems = chain_elems; c->nb = nb; c->n_slots = n_slots;
  }
  CU(c, cudaMemsetAsync(c->slots, 0, sizeof(double) * (size_t)nb * n_slots, c->stream));
  return KBP_OK;
}

static int check_range(kbp_ctx* c, int chain, int64_t off, int64_t n) {
  if (!c || !c->arena) return fail(c, KBP_E_ARG, "arena not reserved");
  if (off < 0 || n < 0 || off + n > c->chain_elems || chain < -1 || chain >= c->nb) return fail(c, KBP_E_ARG, "transfer out of range");
  return KBP_OK;
}

int kbp_upload(kbp_ctx* c, int chain, int64_t off, const void* host, int64_t n) {
  int r = check_range(c, chain, off, n);
  if (r) return r;
  if (n == 0) return KBP_OK;
  CU(c, cudaSetDevice(c->device));
  if (chain >= 0) {
    CU(c, cudaMemcpyAsync(c->arena + (size_t)chain * c->chain_elems + off, host, sizeof(double2) * n, cudaMemcpyHostToDevice, c->stream));
  } else {
    CU(c, cudaMemcpy2DAsync(c->arena + off, sizeof(double2) * c->chain_elems, host, sizeof(double2) * n, sizeof(double2) * n, c->nb,
                            cudaMemcpyHostToDevice, c->stream));
  }
  return KBP_OK;
}

int kbp_broadcast(kbp_ctx* c, int64_t off, const void* host, int64_t n) {
  int r = check_range(c, 0, off, n);
  if (r) return r;
  if (n == 0) return KBP_OK;
  CU(c, cudaSetDevice(c->device));
  // pitch 0 on the source side repeats the same row for every chain
  for (int b = 0; b < c->nb; ++b)
    CU(c, cudaMemcpyAsync(c->arena + (size_t)b * c->chain_elems + off, host, sizeof(double2) * n, cudaMemcpyHostToDevice, c->stream));
  return KBP_OK;
}

int kbp_download(kbp_ctx* c, int chain, int64_t off, void* host, int64_t n) {
  int r = check_range(c, chain, off, n);
  if (r) return r;
  if (n == 0) return KBP_OK;
  CU(c, cudaSetDevice(c->device));
  if (chain >= 0) {
    CU(c, cudaMemcpyAsync(host, c->arena + (size_t)chain * c->chain_elems + off, sizeof(double2) * n, cudaMemcpyDeviceToHost, c->stream));
  } else {
    CU(c, cudaMemcpy2DAsync(host, sizeof(double2) * n, c->arena + off, sizeof(double2) * c->chain_elems, sizeof(double2) * n, c->nb,
                            cudaMemcpyDeviceToHost, c->stream));
  }
  CU(c, ctx_wait(c));
  return KBP_OK;
}

int kbp_slots_read(kbp_ctx* c, double* host) {
  if (!c || !c->slots) return fail(c, KBP_E_ARG, "arena not reserved");
  CU(c, cudaSetDevice(c->device));
  CU(c, cudaMemcpyAsync(host, c->slots, sizeof(double) * (size_t)c->nb * c->n_slots, cudaMemcpyDeviceToHost, c->stream));
  CU(c, ctx_wait(c));
  return KBP_OK;
}

int kbp_slots_zero(kbp_ctx* c) {
  if (!c || !c->slots) return fail(c, KBP_E_ARG, "arena not reserved");
  CU(c, cudaSetDevice(c->device));
  CU(c, cudaMemsetAsync(c->slots, 0, sizeof(double) * (size_t)c->nb * c->n_slots, c->stream));
  return KBP_OK;
}

/* device addresses for zero-copy interoperation with NCCL / torch (multi-GPU exchange of messages between arenas) */
uint64_t kbp_arena_ptr(const kbp_ctx* c) { return c ? (uint64_t)(uintptr_t)c->arena : 0; }
uint64_t kbp_slots_ptr(const kbp_ctx* c) { return c ? (uint64_t)(uintptr_t)c->slots : 0; }
uint64_t kbp_stream_ptr(const kbp_ctx* c) { return c ? (uint64_t)(uintptr_t)c->stream : 0; }
int64_t kbp_chain_elems(const kbp_ctx* c) { return c ? c->chain_elems : 0; }

int kbp_sync(kbp_ctx* c) {
  if (!c) return KBP_E_ARG;
  CU(c, cudaSetDevice(c->device));
  CU(c, ctx_wait(c));
  return KBP_OK;
}

int64_t kbp_svd_work_elems(int64_t m, int64_t n) { return kbp::svd_work_elems(m, n); }
int64_t kbp_qr_work_elems(int64_t m, int64_t n) {
  int64_t k = m < n ? m : n;
  return m * n + m * k + k + 8;
}
int64_t kbp_svd_warm_elems(int64_t, int64_t, int64_t) { return 0; }
int64_t kbp_launch_count(const kbp_ctx* c) { return c ? c->launches : 0; }
double kbp_gemm_flops(const kbp_ctx* c) { return c ? c->gemm_flops : 0.0; }
int kbp_svd_counters(kbp_ctx* c, int64_t* out8) {
  if (!c || !out8) return KBP_E_ARG;
  cudaSetDevice(c->device);
  fold_device_counters(c);                 // synchronises the context's stream
  for (int i = 0; i < 8; ++i) out8[i] = c->counters[i];
  return KBP_OK;
}

int kbp_graph_counters(const kbp_ctx* c, int64_t* out4) {
  if (!c || !out4) return KBP_E_ARG;
  out4[0] = c->graph_replays;
  out4[1] = c->graph_captures;
  int64_t ok = 0, bad = 0;
  for (auto& kv : c->graphs) { ok += kv.second.exec != nullptr; bad += kv.second.bad; }
  out4[2] = ok;
  out4[3] = bad;
  return KBP_OK;
}

int64_t kbp_svd_sweeps(kbp_ctx* c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  fold_device_counters(c);
  return c->counters[5] + c->counters[6];
}

int kbp_timer_start(kbp_ctx* c) {
  if (!c) return KBP_E_ARG;
  CU(c, cudaSetDevice(c->device));
  CU(c, cudaEventRecord(c->ev0, c->stream));
  return KBP_OK;
}

int kbp_timer_stop_ms(kbp_ctx* c, double* ms) {
  if (!c || !ms) return KBP_E_ARG;
  CU(c, cudaSetDevice(c->device));
  CU(c, cudaEventRecord(c->ev1, c->stream));
  CU(c, cudaEventSynchronize(c->ev1));
  float f = 0.f;
  CU(c, cudaEventElapsedTime(&f, c->ev0, c->ev1));
  *ms = f;
  return KBP_OK;
}

int kbp_profile_enable(kbp_ctx* c, int on) {
  if (!c) return KBP_E_ARG;
  c->profile = on != 0;
  return KBP_OK;
}

int kbp_profile_read(kbp_ctx* c, double* ms16, int64_t* count16) {
  if (!c || !ms16 || !count16) return KBP_E_ARG;
  CU(c, cudaSetDevice(c->device));
  CU(c, ctx_wait(c));
  for (auto& sp : c->spans) {
    float f = 0.f;
    if (cudaEventElapsedTime(&f, sp.a, sp.b) == cudaSuccess && sp.op >= 0 && sp.op < 16) { c->prof_ms[sp.op] += f; c->prof_n[sp.op] += 1; }
    cudaEventDestroy(sp.a);
    cudaEventDestroy(sp.b);
  }
  c->spans.clear();
  for (int i = 0; i < 16; ++i) { ms16[i] = c->prof_ms[i]; count16[i] = c->prof_n[i]; c->prof_ms[i] = 0; c->prof_n[i] = 0; }
  return KBP_OK;
}

static inline double bits_to_double(int64_t b) {
  double d;
  memcpy(&d, &b, sizeof(d));
  return d;
}

static int run_ops(kbp_ctx* c, const int64_t* w, int64_t n_words, bool capture, cudaGraph_t top_graph, uint64_t phash);

static uint64_t program_hash(const int64_t* w, int64_t n_words) {
  uint64_t h = 1469598103934665603ull;
  for (int64_t i = 0; i < n_words; ++i) { h ^= (uint64_t)w[i]; h *= 1099511628211ull; }
  return h ^ ((uint64_t)n_words * 0x9E3779B97F4A7C15ull);
}

static const size_t KBP_GRAPH_MAX = 256;

int kbp_graph_policy(kbp_ctx* c, int64_t min_words, int capture_first) {
  if (!c || min_words < 0) return KBP_E_ARG;
  c->graph_min_words = min_words;
  c->graph_first = capture_first != 0;
  return KBP_OK;
}

// 1: the next kbp_run of this program is a single graph launch (asynchronous, no host decisions);  0: it will be run
// op by op with host-driven loops (first sight of the program, graphs disabled, profiling)
int kbp_graph_ready(kbp_ctx* c, const int64_t* w, int64_t n_words) {
  if (!c || !w || !kbp::graphs_enabled() || c->profile || n_words < c->graph_min_words) return 0;
  auto it = c->graphs.find(program_hash(w, n_words));
  if (it == c->graphs.end()) return c->graph_first && c->graphs.size() < KBP_GRAPH_MAX;
  return !it->second.bad && (it->second.exec != nullptr || it->second.seen >= 1 || c->graph_first);
}

// launch the graph of a captured program and count its launches, GEMM flops and host-decided SVD routes
static int launch_graph(kbp_ctx* c, const kbp_ctx::GraphEntry& ge) {
  CU(c, cudaGraphLaunch(ge.exec, c->stream));
  c->launches += ge.launches;
  c->gemm_flops += ge.flops;
  for (int k = 0; k < 2; ++k) c->counters[k] += ge.dcount[k];
  ++c->graph_replays;
  return KBP_OK;
}

// Every program is a CUDA graph from its second run on: the op stream is a constant launch sequence except for the
// truncated SVDs, whose data-dependent loops are captured as conditional WHILE / IF nodes driven by one-thread decision
// kernels (k_tsvd.cu, k_svd.cu).  The first run is host-driven (plain launches, control block read back per decision): it
// validates the program and serves profilers, which want plain launches.
int kbp_run(kbp_ctx* c, const int64_t* w, int64_t n_words) {
  if (!c || !c->arena || !w) return fail(c, KBP_E_ARG, "kbp_run: arena not reserved");
  static const bool graphs_on = kbp::graphs_enabled();
  static const bool sync_every = getenv("KBP_SYNC_EVERY_OP") != nullptr;
  const uint64_t h = program_hash(w, n_words);
  if (!graphs_on || c->profile || sync_every || n_words < c->graph_min_words) return run_ops(c, w, n_words, false, nullptr, h);
  auto it = c->graphs.find(h);
  if (it == c->graphs.end()) {
    if (c->graphs.size() >= KBP_GRAPH_MAX) return run_ops(c, w, n_words, false, nullptr, h);
    it = c->graphs.emplace(h, kbp_ctx::GraphEntry()).first;
  }
  kbp_ctx::GraphEntry& ge = it->second;
  CU(c, cudaSetDevice(c->device));
  if (ge.exec) return launch_graph(c, ge);
  if (ge.bad || (ge.seen++ == 0 && !c->graph_first)) return run_ops(c, w, n_words, false, nullptr, h);
  const int64_t l0 = c->launches;
  const double f0 = c->gemm_flops;
  int64_t c0[8];
  for (int k = 0; k < 8; ++k) c0[k] = c->counters[k];
  auto restore_counters = [&] {
    c->launches = l0;
    c->gemm_flops = f0;
    for (int k = 0; k < 8; ++k) c->counters[k] = c0[k];
  };
  auto give_up = [&](const char* why) {
    ge.bad = true;
    cudaGetLastError();
    restore_counters();
    fprintf(stderr, "[kbp] graph capture of a %lld-word program failed (%s): running it with host-driven loops\n", (long long)n_words, why);
    return run_ops(c, w, n_words, false, nullptr, h);
  };
  // One graph per program.  Cutting a program into graphs of a few thousand launches was measured to be far WORSE: the launch
  // call of the second graph on a stream blocks the host while the first is executing (N = 6 block: 226 ms per call instead
  // of 20-30 ms; six sides 1574 ms instead of 685 ms per BP iteration).
  if (n_words == 0) return give_up("empty program");
  if (cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) return give_up("begin capture");
  cudaStreamCaptureStatus st;
  unsigned long long id;
  cudaGraph_t top = nullptr;
  const cudaGraphNode_t* deps = nullptr;
  size_t nd = 0;
  int rc = KBP_E_CUDA;
  if (cudaStreamGetCaptureInfo_v2(c->stream, &st, &id, &top, &deps, &nd) == cudaSuccess && top) rc = run_ops(c, w, n_words, true, top, h);
  cudaGraph_t graph = nullptr;
  const cudaError_t e1 = cudaStreamEndCapture(c->stream, &graph);
  if (rc != KBP_OK || e1 != cudaSuccess || !graph) {
    for (int k = 0; k < 2; ++k) {                        // a body capture left open by a failure inside an op
      cudaStreamCaptureStatus bs;
      if (cudaStreamIsCapturing(c->body_stream[k], &bs) == cudaSuccess && bs != cudaStreamCaptureStatusNone) { cudaGraph_t g2 = nullptr; cudaStreamEndCapture(c->body_stream[k], &g2); }
    }
    if (graph) cudaGraphDestroy(graph);
    return give_up(rc != KBP_OK ? c->err.c_str() : cudaGetErrorString(e1));
  }
  cudaGraphExec_t ex = nullptr;
  const cudaError_t e2 = cudaGraphInstantiate(&ex, graph, 0);
  cudaGraphDestroy(graph);
  if (e2 != cudaSuccess) return give_up(cudaGetErrorString(e2));
  ge.exec = ex;
  ge.launches = c->launches - l0;
  ge.flops = c->gemm_flops - f0;
  for (int k = 0; k < 8; ++k) ge.dcount[k] = c->counters[k] - c0[k];
  restore_counters();                                    // capturing ran nothing: launch_graph counts the first run
  ++c->graph_captures;
  return launch_graph(c, ge);
}

/* developer probe (KBP_KTIME=1): prints and resets the in-kernel timing of the Cholesky CTAs (k_tsvd.cu) */
int kbp_ktime_report(kbp_ctx* c, const char* tag) {
  if (!c) return KBP_E_ARG;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  kbp::ktime_report(tag ? tag : "");
  return KBP_OK;
}

static int run_ops(kbp_ctx* c, const int64_t* w, int64_t n_words, bool capture, cudaGraph_t top_graph, uint64_t phash) {
  if (!c || !c->arena || !w) return fail(c, KBP_E_ARG, "kbp_run: arena not reserved");
  CU(c, cudaSetDevice(c->device));
  kbp::Arena a;
  a.base = c->arena; a.chain_stride = c->chain_elems; a.slots = c->slots; a.n_slots = c->n_slots; a.nb = c->nb;
  a.stream = c->stream; a.block_event = c->block_event; a.launches = &c->launches; a.gemm_flops = &c->gemm_flops; a.counters = c->counters; a.svd_off = c->svd_off; a.svd_off_host = c->svd_off_host;
  a.scratch = c->scratch; a.scratch_stride = KBP_GEMM_SCRATCH; a.counters_dev = c->counters_dev;
  a.ctl = c->ctl; a.ctl_host = c->ctl_host; a.chain_state = reinterpret_cast<int*>(c->ctl + 1);
  a.mask = nullptr; a.mask_want = 0;
  a.tsvd_rounds = &c->tsvd_rounds; a.op_key = 0;
  a.capture = capture; a.top_graph = top_graph; a.body_stream[0] = c->body_stream[0]; a.body_stream[1] = c->body_stream[1]; a.depth = 0;
  const int64_t E = c->chain_elems;
  auto in_arena = [&](int64_t off, int64_t n) { return off >= 0 && n >= 0 && off + n <= E; };
  auto slot_ok = [&](int64_t s) { return s >= -1 && s < c->n_slots; };
  int64_t i = 0;
  const int status = KBP_OK;
  static const bool sync_every = getenv("KBP_SYNC_EVERY_OP") != nullptr;
  while (i < n_words) {
    const int64_t op = w[i];
    char where[64];
    snprintf(where, sizeof(where), " (op %lld at word %lld)", (long long)op, (long long)i);
#define NEED(k) if (i + 1 + (k) > n_words) return fail(c, KBP_E_PROGRAM, std::string("truncated program") + where)
#define BAD(msg) return fail(c, KBP_E_PROGRAM, std::string(msg) + where)
    cudaEvent_t pa = nullptr, pb = nullptr;
    if (c->profile && !capture) { cudaEventCreate(&pa); cudaEventCreate(&pb); cudaEventRecord(pa, c->stream); }
    switch (op) {
      case KBP_OP_PERMUTE: {
        NEED(4);
        const int64_t dst = w[i + 1], src = w[i + 2], cj = w[i + 3], nd = w[i + 4];
        if (nd < 1 || nd > 8) BAD("permute: ndim must be 1..8");
        NEED(4 + 2 * nd);
        const int64_t* dims = w + i + 5;
        const int64_t* perm = dims + nd;
        int64_t tot = 1;
        bool seen[8] = {false};
        for (int d = 0; d < nd; ++d) {
          tot *= dims[d];
          if (perm[d] < 0 || perm[d] >= nd || seen[perm[d]]) BAD("permute: bad permutation");
          seen[perm[d]] = true;
        }
        if (!in_arena(dst, tot) || !in_arena(src, tot)) BAD("permute: buffer out of arena");
        kbp::permute(a, dst, src, (int)cj, (int)nd, dims, perm);
        i += 5 + 2 * nd;
        break;
      }
      case KBP_OP_GEMM: {
        NEED(8);
        const int64_t C = w[i + 1], A = w[i + 2], B = w[i + 3], m = w[i + 4], n = w[i + 5], k = w[i + 6], oa = w[i + 7], ob = w[i + 8];
        if (m < 0 || n < 0 || k < 0 || oa < 0 || oa > 3 || ob < 0 || ob > 3) BAD("gemm: bad argument");
        if (!in_arena(C, m * n) || !in_arena(A, m * k) || !in_arena(B, k * n)) BAD("gemm: buffer out of arena");
        kbp::gemm(a, C, A, B, m, n, k, (int)oa, (int)ob);
        i += 9;
        break;
      }
      case KBP_OP_QR: {
        NEED(6);
        const int64_t A = w[i + 1], Q = w[i + 2], R = w[i + 3], wk = w[i + 4], m = w[i + 5], n = w[i + 6];
        if (m <= 0 || n <= 0) BAD("qr: bad shape");
        const int64_t k = m < n ? m : n;
        if (!in_arena(A, m * n) || !in_arena(Q, m * k) || !in_arena(R, k * n) || !in_arena(wk, kbp_qr_work_elems(m, n)))
          BAD("qr: buffer out of arena");
        kbp::qr(a, A, Q, R, wk, m, n);
        i += 7;
        break;
      }
      case KBP_OP_SVD: {
        NEED(11);
        a.op_key = phash ^ (0x9E3779B97F4A7C15ull * (unsigned long long)(i + 1));
        const int64_t A = w[i + 1], US = w[i + 2], Vh = w[i + 3], wk = w[i + 4], m = w[i + 5], n = w[i + 6], keep = w[i + 7];
        const int64_t nrb = w[i + 8], s0 = w[i + 9], s1 = w[i + 10], warm = w[i + 11];
        if (m <= 0 || n <= 0 || keep <= 0 || keep > (m < n ? m : n) || !slot_ok(s0) || !slot_ok(s1)) BAD("svd: bad argument");
        if (!in_arena(A, m * n) || !in_arena(US, m * keep) || !in_arena(Vh, keep * n) || !in_arena(wk, kbp::svd_work_elems(m, n)))
          BAD("svd: buffer out of arena");
        (void)warm;                                    // reserved word of the op (no persistent basis any more)
        const int sw = kbp::svd_truncate(a, A, US, Vh, wk, m, n, keep, (int)nrb, (int)s0, (int)s1);
        if (sw < 0) return fail(c, KBP_E_CUDA, std::string("svd: ") + cudaGetErrorString(cudaGetLastError()) + where);
        i += 12;
        break;
      }
      case KBP_OP_NORMALIZE: {
        NEED(3);
        if (!in_arena(w[i + 1], w[i + 2]) || !slot_ok(w[i + 3])) BAD("normalize: bad argument");
        kbp::normalize(a, w[i + 1], w[i + 2], (int)w[i + 3]);
        i += 4;
        break;
      }
      case KBP_OP_EMBED: {
        NEED(11);
        const int64_t dst = w[i + 1], src = w[i + 2], d0 = w[i + 5], d1 = w[i + 6], d2 = w[i + 7], s0 = w[i + 8], s1 = w[i + 9], s2 = w[i + 10];
        if (d0 < 0 || d1 < 0 || d2 < 0 || !slot_ok(w[i + 11])) BAD("embed: bad argument");
        if (d0 * d1 * d2 > 0) {
          const int64_t last = (d0 - 1) * s0 + (d1 - 1) * s1 + (d2 - 1) * s2;
          if (!in_arena(src, d0 * d1 * d2) || dst < 0 || s0 < 0 || s1 < 0 || s2 < 0 || dst + last >= E) BAD("embed: buffer out of arena");
        }
        kbp::embed(a, dst, src, bits_to_double(w[i + 3]), bits_to_double(w[i + 4]), d0, d1, d2, s0, s1, s2, (int)w[i + 11]);
        i += 12;
        break;
      }
      case KBP_OP_ZERO: {
        NEED(2);
        if (!in_arena(w[i + 1], w[i + 2])) BAD("zero: buffer out of arena");
        kbp::zero(a, w[i + 1], w[i + 2]);
        i += 3;
        break;
      }
      case KBP_OP_SCALAR_TO_SLOT: {
        NEED(3);
        if (!in_arena(w[i + 1], 1) || !slot_ok(w[i + 2]) || !slot_ok(w[i + 3])) BAD("scalar_to_slot: bad argument");
        kbp::scalar_to_slot(a, w[i + 1], (int)w[i + 2], (int)w[i + 3]);
        i += 4;
        break;
      }
      case KBP_OP_NONFINITE: {
        NEED(3);
        if (!in_arena(w[i + 1], w[i + 2]) || !slot_ok(w[i + 3]) || w[i + 3] < 0) BAD("nonfinite: bad argument");
        kbp::count_nonfinite(a, w[i + 1], w[i + 2], (int)w[i + 3]);
        i += 4;
        break;
      }
      case KBP_OP_EYE: {
        NEED(3);
        if (w[i + 2] < 0 || w[i + 3] < 0 || !in_arena(w[i + 1], w[i + 2] * w[i + 3])) BAD("eye: buffer out of arena");
        kbp::eye(a, w[i + 1], w[i + 2], w[i + 3]);
        i += 4;
        break;
      }
      case KBP_OP_SU: {
        NEED(37);
        const int64_t* v = w + i + 1;
        const int64_t d = v[6], D = v[7];
        if (!kbp::su_supported((int)d, (int)D) || v[8] < 0 || !slot_ok(v[10]) || !slot_ok(v[11]) || !slot_ok(v[12])) BAD("su: bad argument");
        const int64_t elems = d * D * D * D * D, d4 = d * d * d * d;
        if (!in_arena(v[0], elems) || !in_arena(v[1], elems) || !in_arena(v[2], elems) || !in_arena(v[3], 6 * D) || !in_arena(v[4], d4) ||
            !in_arena(v[5], 6 * d4))
          BAD("su: buffer out of arena");
        int seen[3][4] = {{0}};
        for (int b = 0; b < 6; ++b)
          for (int e = 0; e < 2; ++e) {
            const int64_t s = v[13 + 4 * b + 2 * e], l = v[14 + 4 * b + 2 * e];
            if (s < 0 || s > 2 || l < 0 || l > 3 || seen[s][l]++) BAD("su: the bond table must pair every virtual leg exactly once");
          }
        kbp::simple_update(a, v);
        i += 38;
        break;
      }
      default:
        BAD("unknown opcode");
    }
    if (c->profile && !capture) { cudaEventRecord(pb, c->stream); c->spans.push_back({(int)op, pa, pb}); }
    if (sync_every && !capture) {
      cudaError_t e_ = cudaStreamSynchronize(c->stream);
      if (e_ == cudaSuccess) e_ = cudaGetLastError();
      if (e_ != cudaSuccess) return fail(c, KBP_E_CUDA, std::string("fault detected right after") + where + ": " + cudaGetErrorString(e_));
    }
  }
#undef NEED
#undef BAD
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(c, KBP_E_CUDA, std::string("kernel launch: ") + cudaGetErrorString(e));
  return status;
}

}  // extern "C"
