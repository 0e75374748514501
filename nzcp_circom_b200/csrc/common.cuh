// Shared host-side declarations for libnzcp_prover.so (internal; the public C ABI is include/nzcp_prover.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "ec.cuh"

namespace nzcp {

struct CudaError : std::runtime_error {
  explicit CudaError(const std::string& s) : std::runtime_error(s) {}
};

#define NZCP_CUDA(expr)                                                                              \
  do {                                                                                               \
    cudaError_t e__ = (expr);                                                                        \
    if (e__ != cudaSuccess) {                                                                        \
      char b__[512];                                                                                 \
      snprintf(b__, sizeof b__, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(e__), __FILE__,    \
               __LINE__, #expr);                                                                     \
      throw nzcp::CudaError(b__);                                                                    \
    }                                                                                                \
  } while (0)

extern std::atomic<uint64_t> g_launch_count;  // every kernel launch of this library, process-wide
// Launches are also charged to the prover the calling thread is working for (prove_impl points this at the prover's own
// counter for the duration of the call): nzcp_prover_launch_count / bench.py "gpu_launches" are per prover.
extern thread_local std::atomic<uint64_t>* t_launch_sink;
#define NZCP_LAUNCH_CHECK()                                        \
  do {                                                             \
    nzcp::g_launch_count.fetch_add(1);                             \
    if (nzcp::t_launch_sink) nzcp::t_launch_sink->fetch_add(1);    \
    NZCP_CUDA(cudaGetLastError());                                 \
  } while (0)

static inline unsigned div_up(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

HD int ilog2_u64(uint64_t v) {   // v > 0
#ifdef __CUDA_ARCH__
  return 63 - __clzll((long long)v);
#else
  return 63 - __builtin_clzll(v);
#endif
}

HD uint64_t bitrev_bits(uint64_t x, int bits) {
  if (bits == 0) return 0;
#ifdef __CUDA_ARCH__
  return __brevll(x) >> (64 - bits);
#else
  uint64_t r = 0;
  for (int i = 0; i < bits; i++, x >>= 1) r = (r << 1) | (x & 1);
  return r;
#endif
}

// Owner of CUDA device memory, pinned host memory, events and streams.  Each acquire call returns the raw pointer or
// handle, which the caller keeps in plain non-owning fields; the destructor releases everything in reverse order of
// acquisition, ignoring return codes (it runs during unwinding).  Sizes are exactly what the caller asks for.
class CudaResources {
 public:
  CudaResources() = default;
  CudaResources(CudaResources&& o) noexcept { *this = std::move(o); }
  CudaResources& operator=(CudaResources&& o) noexcept {   // a swap: what this held is released with `o`
    items_.swap(o.items_);
    std::swap(device_bytes_, o.device_bytes_);
    return *this;
  }
  ~CudaResources() { release(); }

  template <class T>
  T* device(size_t count) {
    void*& p = slot(kDevice);
    NZCP_CUDA(cudaMalloc(&p, count * sizeof(T)));
    device_bytes_ += count * sizeof(T);
    return static_cast<T*>(p);
  }
  template <class T>
  T* pinned(size_t count) {
    void*& p = slot(kPinned);
    NZCP_CUDA(cudaMallocHost(&p, count * sizeof(T)));
    return static_cast<T*>(p);
  }
  cudaEvent_t event() {
    void*& h = slot(kEvent);
    cudaEvent_t e = nullptr;
    NZCP_CUDA(cudaEventCreate(&e));
    h = e;
    return e;
  }
  cudaStream_t stream() {   // non-blocking: never synchronises with the legacy default stream
    void*& h = slot(kStream);
    cudaStream_t s = nullptr;
    NZCP_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    h = s;
    return s;
  }
  size_t device_bytes() const { return device_bytes_; }   // sum of the device() sizes

 private:
  enum Kind { kDevice, kPinned, kEvent, kStream };
  struct Item { Kind kind; void* h; };
  // The record exists before the resource, so a resource that was created is always released.
  void*& slot(Kind k) {
    items_.push_back({k, nullptr});
    return items_.back().h;
  }
  void release() noexcept {
    for (auto it = items_.rbegin(); it != items_.rend(); ++it) {
      if (!it->h) continue;
      switch (it->kind) {
        case kDevice: cudaFree(it->h); break;
        case kPinned: cudaFreeHost(it->h); break;
        case kEvent: cudaEventDestroy(static_cast<cudaEvent_t>(it->h)); break;
        case kStream: cudaStreamDestroy(static_cast<cudaStream_t>(it->h)); break;
      }
    }
    items_.clear();
    device_bytes_ = 0;
  }
  std::vector<Item> items_;
  size_t device_bytes_ = 0;
};

// Device time on stream st from construction to end(); ms() waits for the end event.  An inactive timer makes no CUDA
// call and reads 0 ms (the host runs of Exec).
struct Timer {
  CudaResources res;
  cudaEvent_t a = nullptr, b = nullptr;
  cudaStream_t st;
  explicit Timer(cudaStream_t s, bool active = true) : st(s) {
    if (!active) return;
    a = res.event();
    b = res.event();
    NZCP_CUDA(cudaEventRecord(a, st));
  }
  void end() {
    if (b) NZCP_CUDA(cudaEventRecord(b, st));
  }
  float ms() {
    float t = 0;
    if (!b) return t;
    NZCP_CUDA(cudaEventSynchronize(b));
    NZCP_CUDA(cudaEventElapsedTime(&t, a, b));
    return t;
  }
  float stop() {
    end();
    return ms();
  }
};

// One thread per index: op(i) for i < n.
template <int THREADS, class Op>
__global__ void __launch_bounds__(THREADS) for_each_kernel(Op op, uint64_t n) {
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) op(i);
}

// Where a per-index step runs: on the device (for_each_kernel on stream 0, memory from CudaResources) or, for the host
// test hooks, in a loop on the CPU over host memory, making no CUDA call at all.  Memory from alloc() lives as long as the
// executor, so a scope that frees its buffers at its end makes an executor of its own.
class Exec {
 public:
  explicit Exec(bool host) : host_(host) {}
  bool host() const { return host_; }

  template <class T>
  T* alloc(size_t count) {
    if (!host_) return res_.device<T>(count);
    host_mem_.emplace_back(new uint4[div_up(count * sizeof(T), sizeof(uint4))]);   // 16-byte aligned, as Fp is
    return reinterpret_cast<T*>(host_mem_.back().get());
  }
  void upload(void* dst, const void* src, size_t bytes) const {
    if (host_) memcpy(dst, src, bytes);
    else NZCP_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
  }
  void download(void* dst, const void* src, size_t bytes) const {
    if (host_) memcpy(dst, src, bytes);
    else NZCP_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
  }
  // op(i) for i < n, n > 0.
  template <int THREADS, class Op>
  void run(uint64_t n, const Op& op) const {
    if (host_) {
      for (uint64_t i = 0; i < n; i++) op(i);
      return;
    }
    for_each_kernel<THREADS><<<div_up(n, THREADS), THREADS>>>(op, n);
    NZCP_LAUNCH_CHECK();
  }
  Timer timer() const { return Timer(0, !host_); }

 private:
  bool host_;
  CudaResources res_;
  std::vector<std::unique_ptr<uint4[]>> host_mem_;
};

G1Affine g1_generator();   // synth.cu: the BN254 generators, Montgomery affine
G2Affine g2_generator();
Fr host_fr_root(int k);    // ntt.cu: ffjavascript's Fr.w[k], Montgomery

// ---------------------------------------------------------------------------------------------- NTT (ntt.cu)
// Tables for one domain size n = 2^log_n (Montgomery-form Fr, device memory).
struct NttDomain {
  int log_n = 0;
  Fr* tw_fwd = nullptr;   // w^j, j < n/2, w = Fr.w[log_n]
  Fr* tw_inv = nullptr;   // w^-j
  Fr* coset_scale = nullptr;  // n^-1 * inc^bitrev(p), p < n   (iNTT scale fused with batchApplyKey)
  Fr* ninv_scale = nullptr;   // unused slot kept for standalone iNTT: single element n^-1 (device)
  unsigned char* tw_lo_fwd = nullptr;   // log_n >= 10: w^(j n/1024), j < 512, padded layout (ntt.cu tw_pad_off): the twiddles
  unsigned char* tw_lo_inv = nullptr;   // of every stage of a 2^10 tile, bulk-copied into shared memory by the low pass
  CudaResources res;
};
void ntt_domain_create(NttDomain* d, int log_n, cudaStream_t st);
// H pipeline on `batch` polynomials laid out back to back (batch * n elements), in place:
//   evaluations on the 2^log_n subgroup (natural order)  ->  evaluations on the coset inc*subgroup (natural order)
void ntt_coset_pipeline(const NttDomain& d, Fr* data, int batch, cudaStream_t st);
// Standalone natural-order transforms (snarkjs Fr.fft / Fr.ifft semantics); `tmp` is an n-element scratch.
void ntt_forward(const NttDomain& d, Fr* data, Fr* tmp, cudaStream_t st);
void ntt_inverse(const NttDomain& d, Fr* data, Fr* tmp, cudaStream_t st);
// h[i] = fromMontgomery(a[i]*b[i] - c[i])
void ntt_join_abc(const Fr* a, const Fr* b, const Fr* c, Fr* h, size_t n, cudaStream_t st);

// ---------------------------------------------------------------------------------------------- R1CS (r1cs.cu)
struct R1csDevice {
  uint32_t n = 0;            // domain size (rows per matrix)
  uint64_t nnz = 0;
  uint32_t* row_ptr = nullptr;  // 2n+1 entries: rows 0..n-1 = A, n..2n-1 = B
  uint32_t* col = nullptr;      // signal index per coefficient
  Fr* val = nullptr;            // coef * R^2 mod r exactly as stored in zkey section 4
  uint32_t* order = nullptr;    // thread t evaluates constraint order[t]: each 128-row block sorted by row length
};
// abc = [A_T | B_T | C_T], each n Montgomery-form Fr.  witness: plain Fr, n_vars entries.
void r1cs_eval(const R1csDevice& m, const Fr* witness, Fr* abc, cudaStream_t st);

// ---------------------------------------------------------------------------------------------- MSM (msm.cu)
// Precomputed window table of one base section (built once per proving key; the bases never change between proofs):
//   pts[w * n_points + i] = 2^(c*w) * P_i   affine Montgomery, (0,0) = infinity
// so that all windows of a scalar feed ONE bucket set and the Horner pass over windows disappears.
struct MsmTable {
  void* pts = nullptr;
  size_t n_points = 0;   // including pad_front leading infinity points
  int c = 0, n_windows = 0;
  bool g2 = false;
  size_t bytes = 0;
  CudaResources res;     // empty for a view over the caller's bases (msm_table_view)
};
int msm_pick_window(size_t n_points);
int msm_num_windows(int c);
int msm_pick_window_free(size_t n_points);
// d_bases: device array of n_src affine points; the table gets pad_front infinity points in front of them.
void msm_table_create(MsmTable* t, const void* d_bases, size_t n_src, size_t pad_front, bool g2, int c, cudaStream_t st);
// "Table" view of raw bases for the table-free path (one window, memory owned by the caller).
void msm_table_view(MsmTable* t, void* d_bases, size_t n_points, bool g2, int c);

static constexpr int kMsmMaxRounds = 3;

// Bucket sort of one scalar vector: signed c-bit digits -> (table index | sign) entries grouped by bucket, cut into
// tasks of <= kTaskLen entries.  Shared by every MSM that uses the same scalars (A, B1, B2, C all use the witness).
struct MsmSort {
  size_t n_points = 0;
  int c = 0, n_windows = 0;
  size_t n_buckets = 0;     // all buckets: group_buckets * n_groups
  size_t group_buckets = 0; // 2^(c-1)
  int n_groups = 1;         // 1: window-table mode (all windows share the buckets); n_windows: table-free mode
  bool table_free = false;  // entries index the raw bases (no window table); window w accumulates into bucket group w
  bool smem_hist = false;   // histogram in shared memory (<= 2^15 buckets) or with global atomics
  uint32_t n_copies = 0;    // private copies of each bucket counter (smem path: one per block)
  uint32_t* counts = nullptr;
  uint32_t* offsets = nullptr;
  uint32_t* cursors = nullptr;
  uint32_t* block_sums = nullptr;  // scratch of the multi-block scan
  uint32_t* entries = nullptr;
  uint32_t* task_off = nullptr;
  uint2* tasks = nullptr;
  uint32_t* flags = nullptr;      // [1] error flags, [2] total tasks, [3] total entries, [4] task length,
                                  // [5] points left after the affine pair rounds (= [3] when rounds == 0)
  uint32_t* flags_host = nullptr; // pinned mirror
  size_t max_tasks = 0;
  size_t scratch_bytes = 0;
  // Batched-affine pair rounds (msm.cu "pair rounds"): round r halves every bucket's point list (ceil(len / 2)) with
  // affine additions that share one field inversion per thread.  round_off[r * (n_buckets + 1) + b] = first slot of
  // bucket b in the round-r point array (r = 0: the entry list itself, compact copy of `offsets`); red_count[b] =
  // points of bucket b after the last round -- what the task list and the XYZZ accumulation then work on.
  int rounds = 0;
  uint32_t* round_off = nullptr;
  uint32_t* red_count = nullptr;
  size_t round_max[kMsmMaxRounds + 1] = {0, 0, 0, 0};   // upper bound of the point count after round r
  CudaResources res;
};
int msm_pick_rounds(size_t n_points, int c);
int msm_pick_rounds_prover(size_t n_points, int c);
void msm_sort_create(MsmSort* s, size_t n_points, int c, int rounds = -1, bool table_free = false);   // rounds < 0: msm_pick_rounds
void msm_sort_launch(MsmSort* s, const Fr* scalars, size_t n_points, cudaStream_t st);
// After the stream drained: throws if the device flagged a scalar >= r.  Returns the number of non-zero digits.
uint32_t msm_sort_check(const MsmSort* s);

// One MSM against a sorted scalar vector: accumulate -> combine -> bucket reduction.
struct MsmRun {
  bool g2 = false;
  void* partial = nullptr;
  void* buckets = nullptr;
  void* marg = nullptr;       // marginal bucket sums M_k[j], k < n_digits, j < 32
  int n_digits = 0;           // base-32 digits of a bucket id
  int n_groups = 1, c = 0;    // bucket groups (table-free: one per window) and window bits, copied from the sort plan
  uint32_t* marg_done = nullptr;   // per (group, digit): marginal blocks finished (self-resetting)
  void* result = nullptr;     // device: the finished sum as one XYZZ point (msm_run_finish_device)
  uint32_t* heavy_list = nullptr;
  uint32_t* heavy_count = nullptr;   // [0] heavy buckets, [1] heavy chunks
  uint32_t* chunk_off = nullptr;
  void* chunk_partial = nullptr;
  void* out = nullptr;        // device: S_0 .. S_{n_digits-1}, T
  void* out_host = nullptr;   // pinned
  cudaEvent_t ev_acc0 = nullptr, ev_acc1 = nullptr;  // around the bucket accumulation (pair rounds + XYZZ kernel)
  void* round_pts[2] = {nullptr, nullptr};   // affine point arrays of the pair rounds (ping-pong)
  void* round_prefix = nullptr;              // prefix products of the shared inversion, [step][thread]
  void* round_ops = nullptr;                 // round 1: the two operands of every addition, staged by the forward pass
  void* round_prod = nullptr;                // per-thread denominator products, inverted in place between the passes
  size_t scratch_bytes = 0;
  CudaResources res;
};
void msm_run_create(MsmRun* r, const MsmSort* sort, bool g2);
void msm_run_launch(MsmRun* r, const MsmSort* sort, const MsmTable* table, cudaStream_t st);
void msm_run_finish_device(MsmRun* r, cudaStream_t st);
void msm_sum_points(const void* d_pts, uint32_t count, bool g2, void* d_result, cudaStream_t st);
G1XYZZ msm_run_finish_g1(const MsmRun* r);
G2XYZZ msm_run_finish_g2(const MsmRun* r);
float msm_run_accumulate_ms(const MsmRun* r);
// standalone.cu: the MSM data path (window table, signed digits, c-bit buckets, `rounds` pair rounds of k additions per
// thread, running-sum reduction) run on the CPU with the kernels' own code; instantiated for Fq and Fq2.  Montgomery affine
// bases, plain scalars (>= r: NZCP_E_RANGE).
template <class F>
XYZZ<F> host_msm_sim(const uint8_t* bases, const uint8_t* scalars, size_t n, int c, int rounds, int k);

}  // namespace nzcp
